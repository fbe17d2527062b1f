#!/usr/bin/env python
# -*- coding: utf-8 -*-
"""
bench.py — gp.compute() + gp.log_likelihood() throughput (N-points/s) for the HODLR path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg3|cfg2|cfg5]
                    [--dump-outputs DIR]

One "step" = one gp.compute(x, yerr) + one gp.log_likelihood(y) on a fixed synthetic data set (SURVEY.md §8d):
    x = sort(U(0, 10*N/1000)) (rng 1234), yerr = 0.1, y = sin(x) + 0.1*N(0,1).
Default workload = BASELINE.json's metric config: Matern32Kernel 1-D, N = 2^18, HODLRSolver(min_size=256, tol=1e-10,
seed=42).  With --gpus N (launched by torchrun, one rank per GPU) the SAME GP (strong scaling, as the metric is quoted)
is sharded by top-level sub-tree.  `--workload cfg5` is BASELINE.json configs[4]: 131072 points PER GPU (N = 2^20 on 8).

Semantics of both arms (DESIGN.md §2): rng_mode = per-node streams, exhausted blocks keep their low-rank factors
(`exhaust=lowrank`).  `--impl reference` times the CPU oracle (oracle/: Eigen-free restatement of george's hodlr.h; the
reference's own _hodlr extension needs Eigen, which is absent) IN THAT SAME MODE on a bounded sample of the workload
(`config.N` says which N; single thread, as the reference is).  The `ours` line carries `same_n`: the CUDA path timed
at the reference arm's N with the same semantics, and the relative difference of the two log-likelihoods there — that
pair is the like-for-like comparison.  `parity_reference_mode` repeats it in the reference's OWN mode (one shared
mt19937, dense storage of exhausted blocks) at a small N.

JSON keys follow the driver contract; extra: roofline{}, cpu_baseline{}, clocks{}, e2e{}, gpu_launches, same_n{},
kernel_ms{}, secondary{cfg2, cfg4}.

`--dump-outputs DIR` writes what the last timed step returned, as float64 arrays of shape (1,): log_likelihood.npy,
log_determinant.npy and dot_solve.npy (y^T K^-1 y) of the device-resident leg, and log_likelihood_e2e.npy of the
public-API leg.  The inputs are seeded, so two builds run with the same arguments can be compared output for output.
Two runs of one build agreed to 4e-16 relative, not bit for bit (B200, 1000 W power limit), so compare with a tolerance.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: nothing is written next to the sources

# FP64 peaks of this pool's B200, BUILDER-measured with tools/fp64_peaks.cu (profiles/fp64_peaks_r01.txt); the
# driver-written MEASURED_PEAKS.json has only HBM and bf16 entries.  cuBLAS dgemm reaches 35.4 TFLOP/s on the same box.
FP64_TENSOR_PEAK_TFLOPS = 37.2   # DMMA.8x8x4 issue-bound
FP64_DFMA_PEAK_TFLOPS = 34.1     # DFMA issue-bound
# FP64 operations the specialised evaluator executes per covariance entry, counted in the SASS of
# a2_eval_kernel<shape> (cuobjdump; DFMA = 2 flop, DMUL/DADD = 1; exp, sqrt and sin are software sequences on this pipe)
EVAL_FLOPS = {"cfg3": 56.0, "cfg2": 40.0, "cfg5": 120.0}
HBM_FALLBACK_GBS = 6650.0
METRIC = "gp.compute+log_likelihood N-points/sec"


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return json.load(fh), "measured"
    except Exception:
        return {"hbm_gbs": HBM_FALLBACK_GBS}, "fallback"


WORKLOADS = {
    # n: size of the GPU arm (cfg5: per GPU); ref_n: the bounded sample the CPU oracle is timed on
    "cfg3": dict(label="Matern32Kernel 1D N=262144 HODLRSolver leaf=256", n=262144, min_size=256, tol=1e-10,
                 ref_n=65536, refmode_n=2048, weak=False),
    "cfg2": dict(label="ExpSquaredKernel 1D N=65536 HODLRSolver tol=1e-10", n=65536, min_size=100, tol=1e-10,
                 ref_n=65536, refmode_n=16384, weak=False),
    "cfg5": dict(label="ExpSquared+ExpSine2 sum kernel 1D N=131072/GPU HODLRSolver tol=1e-10", n=131072, min_size=100,
                 tol=1e-10, ref_n=16384, refmode_n=8192, weak=True),
}


def make_kernel(name):
    from george_b200 import kernels
    if name == "cfg3":
        return 1.0 * kernels.Matern32Kernel(1.0)
    if name == "cfg2":
        return 1.0 * kernels.ExpSquaredKernel(1.0)
    return 1.0 * kernels.ExpSquaredKernel(1.0) + 0.5 * kernels.ExpSine2Kernel(gamma=1.0, log_period=np.log(3.0))


def make_data(n):
    rng = np.random.default_rng(1234)
    x = np.sort(rng.uniform(0, 10 * n / 1000, n))
    yerr = 0.1 * np.ones(n)
    y = np.sin(x) + 0.1 * rng.normal(size=n)
    return x, yerr, y


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index=0):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, universal_newlines=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for row in self.rows:
            parts = [p.strip() for p in row.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            for nm, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------------
# CPU legs (oracle/ = test infrastructure; bench.py may execute it only here: cpu_baseline and --impl reference)
# ---------------------------------------------------------------------------------------------------------------------
def oracle_step(name, n, rng_mode, exhaust):
    """One compute + log-likelihood of the CPU oracle; rng_mode 1 / exhaust 0 = the reference's own algorithm,
    rng_mode 0 / exhaust 1 = the mode of the GPU arm.  Returns (seconds, log-likelihood, kernel evaluations)."""
    import oracle
    from george_b200._spec import flatten
    wl = WORKLOADS[name]
    x, yerr, y = make_data(n)
    spec = flatten(make_kernel(name))
    t0 = time.perf_counter()
    h = oracle.HODLR(spec, x, yerr, min_size=wl["min_size"], tol=wl["tol"], seed=42, rng_mode=rng_mode, exhaust=exhaust)
    ll = -0.5 * (n * np.log(2 * np.pi) + h.log_determinant) - 0.5 * h.dot_solve(y)
    dt = time.perf_counter() - t0
    return dt, ll, h.num_evals


def sample_text(name, n):
    wl = WORKLOADS[name]
    return ("same kernel / min_size / tol / seed / rng_mode=pernode / exhausted_rows=lowrank at N={0}{1}; one thread (the "
            "reference has no threading)".format(n, "" if n == wl["n"] else " (bounded sample of the workload)"))


def run_reference(args):
    wl = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = wl["ref_n"]
    for _ in range(1 if args.warmup > 0 else 0):  # one warm-up pass is enough for a single-threaded CPU code
        oracle_step(args.workload, n, 0, 1)
    times, ll = [], None
    for _ in range(args.steps):
        dt, ll, _ = oracle_step(args.workload, n, 0, 1)
        times.append(dt)
    value = n * len(times) / sum(times)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "points/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times),
        "higher_is_better": True, "scaling": "weak" if wl["weak"] else "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": wl["label"] + " — CPU arm: bounded sample at N={0}".format(n), "N": n,
                   "N_gpu_arm": wl["n"], "min_size": wl["min_size"], "tol": wl["tol"], "seed": 42,
                   "rng_mode": "pernode", "exhausted_rows": "lowrank",
                   "reference_impl": "oracle/ C++ restatement of george hodlr.h (Eigen absent, _hodlr not buildable), "
                                     "run in the GPU arm's mode"},
        "same_config": n == wl["n"], "same_semantics": True,
        "note": "compare with the GPU arm's same_n block (same N, same semantics); points/s of this CPU path FALLS with N "
                "(its cost grows faster than N), so dividing the GPU arm's full-size value by this number understates "
                "the ratio at full size",
        "log_likelihood": ll,
        "cpu_baseline": {"value": value, "unit": "points/s", "cores": 1, "kind": "port", "sample": sample_text(args.workload, n)},
        "e2e": {"value": value, "unit": "points/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------------------
# GPU legs
# ---------------------------------------------------------------------------------------------------------------------
def pinned_array(lib, n):
    from george_b200 import _lib
    p = C.c_void_p()
    _lib.check(lib.bgp_host_alloc_pinned(C.byref(p), n * 8))
    buf = (C.c_double * n).from_address(p.value)
    return np.frombuffer(buf, dtype=np.float64), p


class DeviceLeg(object):
    """compute + log-likelihood through the C ABI with x / yerr / y resident in HBM."""

    def __init__(self, lib, name, n, rng_mode="pernode", exhaust="lowrank", profile=True):
        from george_b200 import _lib
        from george_b200._spec import flatten
        from george_b200.solvers._hodlr import HODLRSolver as Native
        self.lib, self._lib, self.n = lib, _lib, n
        wl = WORKLOADS[name]
        self.spec = flatten(make_kernel(name))
        self.native = Native()
        x, yerr, y = make_data(n)
        self.ptrs = []
        for a in (x, yerr, y):
            p = C.c_void_p()
            _lib.check(lib.bgp_dev_alloc(C.byref(p), a.nbytes))
            _lib.check(lib.bgp_dev_upload(p, _lib.ptr(a), a.nbytes))
            self.ptrs.append(p)
        self.native.set_profiling(profile)
        self.opts = self.native._opts(wl["min_size"], wl["tol"], 42, rng_mode, 0, 0, 1, exhaust)

    def step(self):
        lib, _lib, n = self.lib, self._lib, self.n
        dx, dyerr, dy = self.ptrs
        _lib.check(lib.bgp_hodlr_compute_dev(self.native._ptr, C.byref(self.spec), dx, n, 1, dyerr, C.byref(self.opts)))
        ld, out = C.c_double(), C.c_double()
        _lib.check(lib.bgp_hodlr_log_determinant(self.native._ptr, C.byref(ld)))
        _lib.check(lib.bgp_hodlr_dot_solve_dev(self.native._ptr, dy, C.byref(out)))
        self.last = {"log_determinant": ld.value, "dot_solve": out.value}
        return -0.5 * (n * np.log(2 * np.pi) + ld.value) - 0.5 * out.value

    def close(self):
        for p in self.ptrs:
            self.lib.bgp_dev_free(p)
        self.ptrs = []
        self.native = None


def time_steps(step, steps, warmup, flush_l2, barrier, collect=None):
    """W warm-ups, then K steps each bracketed by CUDA events with the device idle on both sides; L2 flushed between."""
    import torch
    out = None
    for _ in range(warmup):
        out = step()
    barrier()
    t_dev, t_wall = [], []
    for _ in range(steps):
        flush_l2()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        t0 = time.perf_counter()
        out = step()
        torch.cuda.synchronize()
        e1.record()
        e1.synchronize()
        t_wall.append(time.perf_counter() - t0)
        t_dev.append(1e-3 * e0.elapsed_time(e1))
        if collect is not None:
            collect()
    barrier()
    return out, t_dev, t_wall


def dense_secondary(lib, flush_l2, barrier, reps=2):
    """BASELINE.json configs[3]: Matern52 3-D N=32768 BasicSolver (dense Cholesky on the FP64 tensor pipe)."""
    import george_b200 as george
    from george_b200 import kernels, _lib
    n = 32768
    rng = np.random.default_rng(1234)
    x = rng.uniform(0, 1, (n, 3))
    x = x[np.argsort(x[:, 0])]
    yerr = 0.1 * np.ones(n)
    y = np.sin(x.sum(axis=1)) + 0.1 * rng.normal(size=n)
    s = george.BasicSolver(1.0 * kernels.Matern52Kernel(0.5, ndim=3))
    best = None
    for rep in range(reps + 1):
        flush_l2()
        barrier()
        t0 = time.perf_counter()
        s.compute(x, yerr)
        t1 = time.perf_counter()
        q = s.dot_solve(y)
        t2 = time.perf_counter()
        tm = (C.c_double * 2)()
        lib.bgp_dense_last_timing(s._handle.ptr, tm)
        rec = {"compute_wall_ms": 1e3 * (t1 - t0), "dot_solve_wall_ms": 1e3 * (t2 - t1), "build_ms": tm[0], "potrf_ms": tm[1]}
        if rep > 0 and (best is None or rec["compute_wall_ms"] + rec["dot_solve_wall_ms"] < best["compute_wall_ms"] + best["dot_solve_wall_ms"]):
            best = rec
    ll = -0.5 * (n * np.log(2 * np.pi) + s.log_determinant) - 0.5 * q
    peaks, kind = measured_peaks()
    hbm = peaks.get("hbm_gbs", HBM_FALLBACK_GBS)
    tot = 1e-3 * (best["compute_wall_ms"] + best["dot_solve_wall_ms"])
    out = {"workload": "Matern52Kernel 3D N=32768 BasicSolver dense Cholesky", "N": n, "points_per_s": n / tot,
           "ms_per_step": 1e3 * tot, "log_likelihood": ll, "e2e": "host inputs, wall clock (x, yerr, y copied in; scalar out)",
           "build": {"ms": best["build_ms"], "gbs": 8.0 * n * n / (best["build_ms"] * 1e-3) * 1e-9,
                     "frac_hbm": 8.0 * n * n / (best["build_ms"] * 1e-3) * 1e-9 / hbm, "peak_gbs": hbm, "peak_source": kind},
           "potrf": {"ms": best["potrf_ms"], "tflops": n ** 3 / 3.0 / (best["potrf_ms"] * 1e-3) * 1e-12,
                     "frac_dmma": n ** 3 / 3.0 / (best["potrf_ms"] * 1e-3) * 1e-12 / FP64_TENSOR_PEAK_TFLOPS,
                     "peak_tflops": FP64_TENSOR_PEAK_TFLOPS, "peak_source": "builder-measured DMMA issue peak (tools/fp64_peaks.cu)"},
           "solve": {"ms": best["dot_solve_wall_ms"], "hbm_bound_ms": 2 * 8.0 * n * n / 2 / (hbm * 1e9) * 1e3}}
    del s
    # CPU beside it: the same path (kernel-matrix build by the oracle's restated kernel_interface loop + LAPACK through
    # scipy, the reference's BasicSolver.compute) on a bounded sample
    try:
        import oracle
        import scipy.linalg
        from george_b200._spec import flatten
        ns = 4096
        spec = flatten(1.0 * kernels.Matern52Kernel(0.5, ndim=3))
        t0 = time.perf_counter()
        K = oracle.value_symmetric(spec, x[:ns])
        K[np.diag_indices_from(K)] += yerr[:ns] ** 2
        t1 = time.perf_counter()
        cf = scipy.linalg.cholesky(K, lower=False, overwrite_a=True)
        ld = 2 * np.sum(np.log(np.diag(cf)))
        qq = y[:ns] @ scipy.linalg.cho_solve((cf, False), y[:ns])
        t2 = time.perf_counter()
        out["cpu_baseline"] = {"value": ns / (t2 - t0), "unit": "points/s", "kind": "port", "cores": os.cpu_count(),
                               "sample": "N={0}: serial kernel-matrix loop (1 core) {1:.2f} s + LAPACK dpotrf/dpotrs via scipy "
                                         "(default threads) {2:.2f} s; cost grows like N^3".format(ns, t1 - t0, t2 - t1),
                               "log_likelihood": -0.5 * (ns * np.log(2 * np.pi) + ld) - 0.5 * qq}
    except Exception as exc:
        out["cpu_baseline"] = {"error": repr(exc)}
    return out


def dump_outputs(directory, outputs):
    os.makedirs(directory, exist_ok=True)
    for name, v in outputs.items():
        np.save(os.path.join(directory, name + ".npy"), np.array([v], dtype=np.float64))


def run_ours(args):
    import torch
    from george_b200 import _lib, GP, HODLRSolver

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    lib = _lib.load()
    _lib.check(lib.bgp_set_device(local_rank))
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    wl = WORKLOADS[args.workload]
    n = wl["n"] * (world if wl["weak"] else 1)
    kernel = make_kernel(args.workload)
    x, yerr, y = make_data(n)
    exhaust = args.exhaust
    solver_kw = dict(min_size=wl["min_size"], tol=wl["tol"], seed=42, exhaust=exhaust)
    warmup = max(args.warmup, 3)

    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")  # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    def flush_l2():
        flush.zero_()
        torch.cuda.synchronize()

    # ---------------- leg 1: device-resident inputs (value) ----------------
    phases, aca_prof = [], []
    if world == 1:
        leg = DeviceLeg(lib, args.workload, n, "pernode", exhaust, profile=False)
        step_value = leg.step

        def collect():
            phases.append(leg.native.timing())
    else:
        from george_b200.parallel import ShardedHODLRSolver
        sharded = ShardedHODLRSolver(kernel, **solver_kw)

        last = {}

        def step_value():
            sharded.compute(x[:, None], yerr)
            last.update(log_determinant=sharded.log_determinant, dot_solve=sharded.dot_solve(y))
            return -0.5 * (n * np.log(2 * np.pi) + last["log_determinant"]) - 0.5 * last["dot_solve"]
        collect = None

    sampler = ClockSampler(local_rank)
    for _ in range(warmup):
        step_value()
    barrier()
    if rank == 0:
        sampler.start()
    launches0 = lib.bgp_launch_count()
    ll_value, t_steps, t_wall = time_steps(step_value, args.steps, 0, flush_l2, barrier, collect)
    launches = lib.bgp_launch_count() - launches0
    outputs = dict(leg.last if world == 1 else last, log_likelihood=ll_value)
    total = sum(t_steps)
    if dist is not None:
        t = torch.tensor([total], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total = float(t.item())

    if rank == 0:  # (kept on stderr so that a failure in the second leg does not lose the first)
        sys.stderr.write("[bench] value leg: {0:.3f} ms/step over {1} steps, N={2}, world={3}, log-lik {4!r}\n".format(
            1e3 * total / args.steps, args.steps, n, world, ll_value))
        sys.stderr.flush()
    if world > 1:
        # the sharded handle owns tens of GB of factor panels at the largest sizes: release them (back into the stream-ordered
        # pool, where the GP's own handle below finds blocks of the right sizes) before the second leg builds its solver
        sharded.solver = None
        del sharded
        import gc
        gc.collect()
        torch.cuda.synchronize()

    # ---------------- leg 2: end to end through the public GP API with pinned HOST buffers (e2e) ----------------
    hx, px = pinned_array(lib, n)
    hyerr, pyerr = pinned_array(lib, n)
    hy, py = pinned_array(lib, n)
    hx[:] = x; hyerr[:] = yerr; hy[:] = y
    if world == 1:
        gp = GP(kernel, solver=HODLRSolver, **solver_kw)
    else:
        from george_b200.parallel import ShardedHODLRSolver
        gp = GP(kernel, solver=ShardedHODLRSolver, **solver_kw)

    def step_e2e():
        gp.compute(hx, hyerr)
        return gp.log_likelihood(hy)

    ll_e2e, t_e2e, _ = time_steps(step_e2e, args.steps, warmup, flush_l2, barrier)
    total_e2e = sum(t_e2e)
    if dist is not None:
        t = torch.tensor([total_e2e], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_e2e = float(t.item())
    clocks = sampler.stop() if rank == 0 else None
    outputs["log_likelihood_e2e"] = ll_e2e
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    peaks, peaks_kind = measured_peaks()
    value = n * args.steps / total
    e2e_value = n * args.steps / total_e2e
    line = {
        "metric": METRIC, "value": value, "unit": "points/s", "n_gpus": world,
        "steps": args.steps, "warmup": warmup, "ms_per_step": 1e3 * total / args.steps,
        "ms_per_step_wall": 1e3 * sum(t_wall) / args.steps,
        "higher_is_better": True, "scaling": "weak" if wl["weak"] else "strong", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": wl["label"] + (" sharded by top-level sub-tree over {0} GPUs".format(world) if world > 1 else ""),
                   "N": n, "min_size": wl["min_size"], "tol": wl["tol"], "seed": 42, "rng_mode": "pernode",
                   "exhausted_rows": exhaust, "l2": "flushed between timed iterations (256 MB memset)",
                   "timing": "CUDA events bracketing each step (device idle on both sides: the events also cover the host "
                             "gaps of the lock-step loop), summed over the K steps, max over ranks; ms_per_step_wall = host clock"},
        "log_likelihood": ll_value, "log_likelihood_e2e": ll_e2e,
        "e2e": {"value": e2e_value, "unit": "points/s", "h2d_bytes_per_step": 3 * n * 8, "d2h_bytes_per_step": 16,
                "ms_per_step": 1e3 * total_e2e / args.steps, "api": "george_b200.GP.compute + GP.log_likelihood"},
        "gpu_launches": int(launches), "clocks": clocks,
    }
    if world == 1:
        ms_step = 1e3 * total / args.steps
        work = leg.native.work()
        # per-kernel times: a few EXTRA, untimed steps with CUDA events around every launch of the lock-step loop (the
        # timed steps above run the loop as one captured graph, where per-kernel events cannot be placed)
        leg.native.set_profiling(True)
        for _ in range(3):
            flush_l2()
            leg.step()
            aca_prof.append(leg.native.aca_profile())
        leg.native.set_profiling(False)
        kms = {k: statistics.mean(p["kernel_ms"][k] for p in aca_prof) for k in aca_prof[0]["kernel_ms"]}
        ev_ms = kms["a2_eval"]
        launches_eval = statistics.mean(p["eval_launches"] for p in aca_prof)
        verified = statistics.mean(p["evals"] for p in aca_prof)
        evaluated = statistics.mean(p["evaluated"] for p in aca_prof)
        fmas = statistics.mean(p["update_fmas"] for p in aca_prof)
        flops = evaluated * EVAL_FLOPS[args.workload] + 2.0 * fmas
        achieved = flops / (ev_ms * 1e-3) * 1e-12
        traffic = None
        try:  # DRAM bytes of one launch of the kernel from the committed `ncu --set full` capture (read + written)
            import csv
            with open(os.path.join(ROOT, "profiles", "prof_a2_eval_r02_raw.csv")) as fh:
                rows = list(csv.reader(fh))
            hdr, units = rows[0], rows[1]
            scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
            traffic = 0.0
            for name in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                i = hdr.index(name)
                traffic += float(rows[2][i]) * scale[units[i]]
        except Exception:
            traffic = None
        ph = {"leaves_concurrent_with_aca": statistics.mean(p["leaves_ms"] for p in phases),
              "aca": statistics.mean(p["aca_ms"] for p in phases), "upsweep": statistics.mean(p["upsweep_ms"] for p in phases),
              "solve": statistics.mean(p["solve_ms"] for p in phases)}
        line["phases_ms"] = ph
        line["kernel_ms"] = dict(kms, leaves=ph["leaves_concurrent_with_aca"], upsweep=ph["upsweep"], solve=ph["solve"],
                                 note="ACA kernels: CUDA events around every launch of the lock-step loop in 3 extra untimed "
                                      "steps (the timed steps run the loop as one captured graph); leaves / upsweep / solve: "
                                      "device events of the timed steps.  step = max(leaves, aca) + upsweep + solve + host gaps")
        line["roofline"] = {
            "kernel": "a2_eval_kernel", "bound": "fp64_alu",
            "pipe": "FP64 CUDA-core pipe (DFMA/DMUL/DADD; software exp/sqrt; no matrix contraction in this kernel, so neither "
                    "'hbm' nor 'tensor' applies)",
            "achieved": achieved, "peak": FP64_DFMA_PEAK_TFLOPS, "unit": "TFLOP/s", "frac": achieved / FP64_DFMA_PEAK_TFLOPS,
            "traffic": traffic,
            "peak_source": "BUILDER-measured FP64 DFMA issue peak (tools/fp64_peaks.cu on this pool, profiles/fp64_peaks_r01.txt); "
                           "MEASURED_PEAKS.json has no FP64 entry (its hbm_gbs = {0} [{1}]); DMMA peak {2}, cuBLAS dgemm 35.4".format(
                               peaks.get("hbm_gbs"), peaks_kind, FP64_TENSOR_PEAK_TFLOPS),
            "algorithmic_flops_per_launch": flops / launches_eval, "launch_ms": ev_ms / launches_eval,
            "launches_per_step": launches_eval, "entries_verified_per_step": verified,
            "entries_evaluated_per_step": evaluated, "flops_per_eval": EVAL_FLOPS[args.workload],
            "counts": "only EVALUATED entries are charged (entries bounded below the 1e-14 pivot threshold without evaluation "
                      "cost no flops and are not counted)",
            "share_of_step": ev_ms / ms_step}
        line["work"] = work
        leg.close()
        if not args.no_cpu:
            # ---- like-for-like: same N, same semantics, CPU oracle vs CUDA path ----
            ns = wl["ref_n"]
            try:
                cpu_s, cpu_ll, cpu_evals = oracle_step(args.workload, ns, 0, 1)
                line["cpu_baseline"] = {"value": ns / cpu_s, "unit": "points/s", "cores": 1, "kind": "port", "seconds": cpu_s,
                                        "kernel_evals": cpu_evals, "sample": sample_text(args.workload, ns)}
                lg = DeviceLeg(lib, args.workload, ns, "pernode", exhaust, profile=False)
                ll_s, t_s, _ = time_steps(lg.step, 5, 3, flush_l2, barrier)
                lg.close()
                gp2 = GP(kernel, solver=HODLRSolver, **solver_kw)
                xs, yerrs, ys = make_data(ns)

                def step_s():
                    gp2.compute(xs, yerrs)
                    return gp2.log_likelihood(ys)
                ll_s2, t_s2, _ = time_steps(step_s, 5, 3, flush_l2, barrier)
                line["same_n"] = {"N": ns, "semantics": "rng_mode=pernode, exhausted_rows={0} on both sides".format(exhaust),
                                  "gpu_points_per_s": ns * len(t_s) / sum(t_s), "gpu_ms_per_step": 1e3 * sum(t_s) / len(t_s),
                                  "gpu_e2e_points_per_s": ns * len(t_s2) / sum(t_s2), "gpu_e2e_ms_per_step": 1e3 * sum(t_s2) / len(t_s2),
                                  "cpu_points_per_s": ns / cpu_s, "cpu_seconds": cpu_s,
                                  "speedup_same_n_same_semantics": (ns * len(t_s2) / sum(t_s2)) / (ns / cpu_s),
                                  "log_likelihood_gpu": ll_s, "log_likelihood_cpu": cpu_ll,
                                  "rel_err": abs(ll_s - cpu_ll) / abs(cpu_ll), "bar": 1e-6}
            except Exception as exc:  # the check must never cost the bench line
                line["same_n"] = {"N": ns, "error": repr(exc)}
            # ---- the reference's OWN algorithm (shared mt19937, dense storage of exhausted blocks) at a small N ----
            nr = wl["refmode_n"]
            try:
                from george_b200.solvers._hodlr import HODLRSolver as Native
                cpu_s, cpu_ll, _ = oracle_step(args.workload, nr, 1, 0)
                xs, yerrs, ys = make_data(nr)
                chk = Native()
                t_same = None
                for _ in range(2):  # second pass: buffers and capacities are warm, as in the timed legs
                    t0 = time.perf_counter()
                    chk.compute(kernel, xs[:, None], yerrs, wl["min_size"], wl["tol"], 42, rng_mode="reference", exhaust="dense")
                    ll_gpu = -0.5 * (nr * np.log(2 * np.pi) + chk.log_determinant) - 0.5 * chk.dot_solve(ys)
                    t_same = time.perf_counter() - t0
                line["parity_reference_mode"] = {
                    "n": nr, "mode": "rng_mode=reference, exhaust=dense (the reference algorithm, hodlr.h:136-221)",
                    "log_likelihood_gpu": ll_gpu, "log_likelihood_cpu": cpu_ll,
                    "rel_err": abs(ll_gpu - cpu_ll) / abs(cpu_ll), "bar": 1e-6,
                    "gpu_seconds": t_same, "cpu_seconds": cpu_s, "speedup": cpu_s / t_same}
            except Exception as exc:
                line["parity_reference_mode"] = {"n": nr, "error": repr(exc)}
        if not args.no_secondary and args.workload == "cfg3":
            sec = {}
            try:  # configs[1]: ExpSquared N=65536, both arms at FULL size
                lg = DeviceLeg(lib, "cfg2", WORKLOADS["cfg2"]["n"], "pernode", exhaust, profile=False)
                l0 = lib.bgp_launch_count()
                ll2, t2, _ = time_steps(lg.step, 10, 3, flush_l2, barrier)
                l1 = lib.bgp_launch_count()
                lg.close()
                n2 = WORKLOADS["cfg2"]["n"]
                sec["cfg2"] = {"workload": WORKLOADS["cfg2"]["label"], "N": n2, "points_per_s": n2 * len(t2) / sum(t2),
                               "ms_per_step": 1e3 * sum(t2) / len(t2), "gpu_launches_per_step": (l1 - l0) / 13.0,
                               "log_likelihood": ll2}
                if not args.no_cpu:
                    cpu_s, cpu_ll, _ = oracle_step("cfg2", n2, 0, 1)
                    sec["cfg2"]["cpu_baseline"] = {"value": n2 / cpu_s, "unit": "points/s", "cores": 1, "kind": "port",
                                                   "seconds": cpu_s, "sample": sample_text("cfg2", n2), "log_likelihood": cpu_ll}
                    sec["cfg2"]["rel_err_vs_cpu"] = abs(ll2 - cpu_ll) / abs(cpu_ll)
                    sec["cfg2"]["speedup_same_n_same_semantics"] = sec["cfg2"]["points_per_s"] / (n2 / cpu_s)
            except Exception as exc:
                sec["cfg2"] = {"error": repr(exc)}
            try:
                sec["cfg4"] = dense_secondary(lib, flush_l2, barrier)
            except Exception as exc:
                sec["cfg4"] = {"error": repr(exc)}
            line["secondary"] = sec
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS))
    ap.add_argument("--exhaust", default="lowrank", choices=["dense", "lowrank"])
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step of the CUDA path to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
