#!/usr/bin/env python
"""bench.py — CG iterations/s on the BASELINE.json workloads, with roofline and CPU baseline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload sparse_ls|rosenbrock|logreg|batched] [--n N] [--coh C] [--quadratic-ls]
                    [--dump-outputs DIR]

A "step" is one iteration of the `for n = 1:max_iters` body of minimizeobjective
(src/engine/optim.jl:50-160): one strong-Wolfe line search (>= 1 fdf! trial) + getβ + the
state roll + updatedir!.  The workload is BASELINE.json's metric config: sparse least squares
½‖Ax−b‖², CSR A 2e8×2e8 with 10 nnz/row, FP64 Hager-Zhang CG (configs[2]; it fits one B200);
`--workload rosenbrock` runs configs[1] (extended Rosenbrock n = 1e8), `logreg` configs[3] (CSR
logistic regression 5e7 × 2e7, L-BFGS m = 10), `batched` configs[4] (262,144 independent n = 512
problems, whole solver on the device).  Under torchrun the rows / vector slices / samples / problems
are sharded over the ranks (total work fixed: "strong" scaling).

`--impl reference` times the reference's CPU path — oracle/ (the C restatement; Julia is not
installed here or on the GPU box) in the reference's own shape: unfused passes, allocating
getβ, sequential sums — on the host cores, on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FULL_N = {"sparse_ls": 200_000_000, "rosenbrock": 100_000_000, "logreg": 20_000_000, "batched": 512}
SAMPLE_N = {"sparse_ls": 20_000_000, "rosenbrock": 10_000_000, "logreg": 2_000_000, "batched": 512}   # CPU arm: n/10 (BASELINE.md §3)
LOGREG_SAMPLES_PER_FEATURE = 2.5      # cfg 4: 5e7 samples x 2e7 features, 20 nnz/row
BATCHED_NPROB = 262_144               # cfg 5


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--workload", default="sparse_ls", choices=["sparse_ls", "rosenbrock", "logreg", "batched"])
    p.add_argument("--n", type=int, default=0, help="problem size (default: BASELINE.json's)")
    p.add_argument("--coh", type=int, default=0,
                   help="sparse_ls generator: log2 of the number of consecutive rows sharing their column offsets "
                        "(0: every row draws its own nine offsets, the banded-random matrix of SURVEY.md §8d cfg 3 — "
                        "the headline; 30: the same offsets for all rows, i.e. ten true diagonals — reported as "
                        "`secondary` by the default run)")
    p.add_argument("--no-secondary", action="store_true", help="sparse_ls: skip the second matrix variant")
    p.add_argument("--gather-block-mib", type=float, default=0.0,
                   help="logreg: size of the column blocks of the gathered vectors (0: library default, 40 MiB)")
    p.add_argument("--max-reps", type=int, default=100, help="cap on the repetitions of the K-step measurement")
    p.add_argument("--min-timed-s", type=float, default=0.0,
                   help="repeat the K-step measurement (fresh run from x0 each time) until the timed region is this long "
                        "(default 0: one measurement, exactly --steps timed steps)")
    p.add_argument("--no-parity-assert", action="store_true",
                   help="report parity_vs_n1 of the headline variant without failing when it exceeds 1e-10")
    p.add_argument("--write-fixture", action="store_true",
                   help="N = 1: (re)write tests/golden/bench_trace_n1.json, the objective traces `parity_vs_n1` checks against")
    p.add_argument("--reduction-ctas", type=int, default=0, help="canonical-order G (0: library default)")
    p.add_argument("--quadratic-ls", action="store_true",
                   help="sparse_ls only: the quadratic-aware line search (SURVEY.md §8f N1), one SpMV + one SpMVT per iteration")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps, write what the timed path returns after its last step (iterate, gradient, "
                        "objective, trace; a fixed sample of long vectors) as DIR/<name>.npy, so that two builds can be "
                        "compared on the same inputs")
    return p.parse_args()


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: an NVML polling thread
    (5 ms period, so that even a 30 ms region gets samples); falls back to an `nvidia-smi -lms`
    subprocess when pynvml is unavailable.  Only samples taken between mark_begin() and mark_end()
    count."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.p = self.f = self.thread = None
        self.samples = []               # (t, sm_mhz, reasons bitmask)
        self.t_begin = self.t_end = None
        self.max_mhz = None
        self._stop = False

    def _nvml_loop(self, nv, h):
        while not self._stop:
            try:
                self.samples.append((time.perf_counter(), float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)),
                                     int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(h))))
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        try:
            import threading
            import pynvml as nv
            import torch
            nv.nvmlInit()
            uuid = str(torch.cuda.get_device_properties(self.idx).uuid)
            h = nv.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self.nv = nv
            self.thread = threading.Thread(target=self._nvml_loop, args=(nv, h), daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            self.p = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "20"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def mark_begin(self):
        self.t_begin = time.perf_counter()

    def mark_end(self):
        self.t_end = time.perf_counter()

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.thread is not None:
            self._stop = True
            self.thread.join(timeout=2)
            nv = self.nv
            t0 = self.t_begin if self.t_begin is not None else -1e300
            t1 = self.t_end if self.t_end is not None else 1e300
            inside = [s_ for s_ in self.samples if t0 <= s_[0] <= t1]
            how = "inside the timed region"
            if not inside and self.samples:      # region shorter than one polling period
                mid = 0.5 * (t0 + t1)
                inside = sorted(self.samples, key=lambda s_: abs(s_[0] - mid))[:3]
                how = "nearest to the timed region"
            if inside:
                bits = 0
                for s_ in inside:
                    bits |= s_[2]
                names = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                         "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                         "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                         "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
                out = {"sm_mhz": float(np.median([s_[1] for s_ in inside])), "sm_max_mhz": self.max_mhz,
                       "reasons": sorted(k for k, v in names.items() if bits & v), "samples": len(inside),
                       "source": "NVML polling thread, " + how}
            return out
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            c = [t.strip() for t in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2]))
            except ValueError:
                continue
            for nm, v in zip(names, c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                   "samples": len(sm), "source": "nvidia-smi -lms 20"}
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        return out


# ------------------------------------------------------------------------------ workloads
def solver_configs(cg, max_iters, workload="sparse_ls"):
    # examples/min.jl:16-35: HagerZhang, StrongWolfeBisection(c1=1e-5, c2=0.8, growth 2, 1000, 100).
    # ϵ is set far below reach so that W+K iterations always run (the metric is iterations/s).
    if workload == "logreg":          # SURVEY.md §8d cfg 4: LBFGS(m=10) + StrongWolfe(1e-4, 0.9)
        cfg = cg.setupCGConfig(1e-300, cg.LBFGS(10), cg.EnableTrace(), max_iters=max_iters)
        ls = cg.setupStrongWolfeBisection(1e-4, 0.9, a_max_growth_factor=2.0, max_iters=1000, zoom_max_iters=100)
        return cfg, ls
    cfg = cg.setupCGConfig(1e-300, cg.HagerZhang(), cg.EnableTrace(), max_iters=max_iters)
    ls = cg.setupStrongWolfeBisection(1e-5, 0.8, a_max_growth_factor=2.0, max_iters=1000, zoom_max_iters=100)
    return cfg, ls


def make_objective(cg, args, ctx, n):
    if args.workload == "rosenbrock":
        obj = cg.RosenbrockGPU(n, ctx)
        x0 = obj.default_x0(24, 0.1)
    elif args.workload == "logreg":
        obj = cg.LogRegGPU(int(n * LOGREG_SAMPLES_PER_FEATURE), n, 20, 24, 1e-6, ctx)
        x0 = np.zeros(obj.n_local)
    else:
        obj = cg.SparseLSGPU(n, 10, None, 24, args.coh, ctx)
        x0 = np.zeros(obj.n_local)
    return obj, x0


def shard_len(n, world, rank, align=2):
    """length of cgo_shard_range(n, world, rank, align)"""
    units = n // align
    lo = (units * rank // world) * align
    hi = n if rank == world - 1 else (units * (rank + 1) // world) * align
    return hi - lo


def matrix_bytes(n_local, nnz_local):
    """one streaming pass over a CSR matrix: 8 B value + 4 B column index per entry + row pointers"""
    return 12.0 * nnz_local + 8.0 * (n_local + 1)


def algorithmic_bytes(args, n_local, nnz_local, evals, iters):
    """Algorithmic HBM bytes (DESIGN.md §bytes) of `iters` iterations with `evals` fdf! trials on
    one rank: what the fused kernels must move when every vector is read / written once per kernel.
    Rosenbrock: trial R x,g,u W xp,g⁺ = 40n, the first trial of an iteration also W u = 48n.
    CSR least squares, per trial: K_a R x,u W xp = 24n | K_b A + gather xp 8n + R b 8n + W r 8n |
    K_c Aᵀ + gather r 8n + R u,g 16n + W g⁺ 8n  = 2M + 80n; the first trial of an iteration also
    R g, W u in K_a = +16n.  (SURVEY.md §8d's formula, (2M + 72n)·E + 48n, is larger: the β-dot
    pass and the direction pass it counts separately are fused away here.)"""
    if args.workload == "rosenbrock":
        return 8.0 * n_local * (6 * iters + 5 * (evals - iters))
    if args.workload == "logreg":
        # per iteration: K_a of the first trial is unfused (24d), pair staging R 4 vectors W 2 = 48d,
        # two-loop recursion with m = 10: 8d(4m + 3) (DESIGN.md)
        per_eval, _ = logreg_bytes(args, n_local, nnz_local)
        return evals * per_eval + iters * (48.0 * n_local + 8.0 * n_local * 43)
    per_eval = 2 * matrix_bytes(n_local, nnz_local) + 80.0 * n_local
    return evals * per_eval + 16.0 * n_local * iters


def ncu_traffic(args, world, n, coh=None):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture of this very
    configuration (profiles/, taken with the commands in scratch/profile_r1.sh, scratch/gpu_r2_ncu_final.sh); None for
    any other configuration."""
    coh = args.coh if coh is None else coh
    name = {"sparse_ls": ("r1_ncu_full_ls_r1b.txt", 200_000_000), "rosenbrock": ("r1_ncu_full_rosen_r1.txt", 100_000_000)}
    if args.workload == "sparse_ls" and coh == 0:
        name["sparse_ls"] = ("r2_ncu_full_sparse_ls_coh0_n2e8_k_spmv_direct.txt", 200_000_000)
    if world != 1 or args.workload not in name or n != name[args.workload][1] or (args.workload == "sparse_ls" and 0 < coh < 28):
        return None, None
    path = os.path.join(ROOT, "profiles", name[args.workload][0])
    try:
        rd, wr = [], []
        for line in open(path):
            t = line.split()
            if len(t) >= 3 and t[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                v = float(t[1]) * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}[t[2]]
                (rd if t[0].endswith("read.sum") else wr).append(v)
        if not rd or len(rd) != len(wr):
            return None, None
        return round(sum(r + w for r, w in zip(rd, wr)) / len(rd), 1), \
            f"bytes per launch, mean of {len(rd)} launches: dram__bytes_read.sum + dram__bytes_write.sum, profiles/{name[args.workload][0]}"
    except OSError:
        return None, None


def logreg_bytes(args, d_loc, nnz_loc):
    """(algorithmic bytes of one fdf! on this rank, of which the K_b + K_c launch pair)
    one rank:  K_a 24d | K_b A + gather w 8d + R y 8N + W c 8N | K_c Aᵀ + gather c 8N + R u,g,w 24d + W g⁺ 8d
    R ranks:   K_a 24d_loc | K_b A_r + gather w 8d + R y, W c 16N_loc | K_c Aᵀ_r + gather c 8N_loc + W part 8d |
               combine R (R parts + u,g,w) W g⁺ = 8d_loc(R + 4)   (exchanges travel over NVLink, not HBM-counted)"""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    d = args.n or FULL_N["logreg"]
    N_loc = nnz_loc // 20
    mats = (12.0 * nnz_loc + 8.0 * (N_loc + 1)) + (12.0 * nnz_loc + 8.0 * (d + 1))
    if world == 1:
        pair = mats + 40.0 * d + 24.0 * N_loc
        return pair + 24.0 * d, pair
    pair = mats + 16.0 * d + 24.0 * N_loc
    return pair + 24.0 * d_loc + 8.0 * d_loc * (world + 4), pair


FIXTURE = os.path.join(ROOT, "tests", "golden", "bench_trace_n1.json")


def workload_text(args, n, coh):
    if args.workload == "sparse_ls":
        return (f"sparse least-squares 0.5||Ax-b||^2, CSR {n}x{n}, 10 nnz/row (banded, |col-row| < 2^20, seed 24, coh_log2={coh}: "
                + ("the same nine offsets for all rows = ten diagonals" if coh >= 28 else
                   ("every row draws its own nine offsets (banded-random, SURVEY.md §8d cfg 3)" if coh == 0 else
                    "offsets redrawn every 2^%d rows" % coh))
                + "), Hager-Zhang CG + StrongWolfeBisection(1e-5,0.8)")
    if args.workload == "logreg":
        return (f"CSR logistic regression {int(n * LOGREG_SAMPLES_PER_FEATURE)} samples x {n} features, "
                f"20 nnz/row, lambda 1e-6, L-BFGS m=10 + StrongWolfeBisection(1e-4,0.9)")
    return f"extended Rosenbrock n={n}, Hager-Zhang CG + StrongWolfeBisection(1e-5,0.8)"


def fixture_key(args, n, coh):
    return f"{args.workload}/n={n}" + (f"/coh={coh}" if args.workload == "sparse_ls" else "") + \
        ("/quadratic" if args.quadratic_ls else "")


def parity_vs_n1(args, n, coh, trace):
    """max relative difference between this run's objective trace (iterations 1…) and the committed N = 1 trace of
    the same configuration (tests/golden/bench_trace_n1.json): the driver-visible 1-vs-N check of SURVEY.md §4 vi."""
    try:
        with open(FIXTURE) as f:
            ref = json.load(f)["traces"].get(fixture_key(args, n, coh))
    except (OSError, ValueError, KeyError):
        ref = None
    if not ref:
        return None, "no fixture for this configuration"
    ref = np.array([float.fromhex(v) for v in ref])
    k = min(len(ref), len(trace))
    if k == 0:
        return None, "empty trace"
    rel = np.abs(np.asarray(trace[:k]) - ref[:k]) / np.abs(ref[:k])
    bad = np.nonzero(rel > PARITY_TOL)[0]
    within = int(bad[0]) if bad.size else k
    return float(rel.max()), f"first {k} iterations; within {PARITY_TOL:g} over the first {within}"


PARITY_TOL = 1e-10      # north_star's gate on per-iteration f (SURVEY.md §8d "Parity gates")


def parity_gate(args, par, what):
    """The headline variant must reproduce the committed one-GPU trace to PARITY_TOL at every rank count (its
    reductions are deterministic for a fixed N, so this either always holds or never does)."""
    if par is not None and par > PARITY_TOL and not args.no_parity_assert:
        raise AssertionError(f"{what}: objective trace differs from the N = 1 fixture by {par:.3e} > {PARITY_TOL:g} "
                             f"(--no-parity-assert reports it without failing)")


DUMP_ENTRIES = 1 << 19        # --dump-outputs: entries kept of a longer output vector (4 MiB in float64)
DUMP_LIMIT = 64 << 20         # --dump-outputs: bytes written at most, all files and ranks together


def sample_index(n, cap):
    """Sorted indices of the entries --dump-outputs keeps of an output of length n: all of them when n <= cap,
    else cap of them drawn with a fixed seed, so that every run with the same arguments keeps the same ones."""
    if n <= cap:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, cap, replace=False))


def run_outputs(run, cap):
    """What a caller of the timed path holds after its last step: the iterate and the gradient (`Results.minimizer`,
    `.gradient`: this rank's shard, sampled), f there, and the trace of the run up to that step."""
    ret = run.results()
    idx = sample_index(len(ret.minimizer), cap)
    k, t = run.n, ret.trace
    return {"minimizer": ret.minimizer[idx], "gradient": ret.gradient[idx], "sample_index": idx,
            "objective": np.array([run.f_x]), "trace_objective": t.objective[:k], "trace_grad_norm": t.grad_norm[:k],
            "trace_step_size": t.step_size[:k], "trace_objective_evals": t.objective_evals[:k]}


def write_outputs(path, arrays, rank, world):
    """path/<name>.npy (path/<name>_rank<r>.npy under torchrun), in float64 unless the output is float32"""
    out = {k: np.asarray(v, dtype=np.float32 if np.asarray(v).dtype == np.float32 else np.float64)
           for k, v in arrays.items()}
    size = world * sum(a.nbytes for a in out.values())
    assert size <= DUMP_LIMIT, f"--dump-outputs: {size} bytes > {DUMP_LIMIT}"
    os.makedirs(path, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(path, k + (f"_rank{rank}" if world > 1 else "") + ".npy"), a)


def measure_device(cg, torch, args, ctx, obj, x0, n, coh, world, rank, local_rank, stream, barrier, dump=False):
    """Device-resident throughput of one configuration: W untimed iterations, then EXACTLY K timed ones (CUDA
    events on the ctx stream), repeated from x0 until the timed region is at least --min-timed-s long (by default
    once); `ms` is the mean over the repetitions.  `dump`: also return what the run holds after the last timed
    step (run_outputs), read after the clock stopped.
    The metric is iterations/s with ϵ out of reach, so a run only ends when the
    line search hits the FP64 floor of the objective (≈53 iterations on cfg 3, ≈28 on cfg 4: both problems are
    well conditioned).  If that happens inside a repetition, the clock stops at the end of the last completed
    iteration (the 100-trial zoom that fails is not an iteration and is not timed) and a fresh run continues the
    count from x0.  With W + K <= 50 this never triggers on cfg 3."""
    K, W = max(args.steps, 1), max(args.warmup, 3)       # timing rule: at least three warm-up steps
    cfg, ls = solver_configs(cg, W + K + 1, args.workload)
    qkw = {"quadratic_linesearch": True} if (args.quadratic_ls and args.workload == "sparse_ls") else {}
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()          # polling runs through the warm-up; only the timed window is reported
    reps, ms_tot, wall_tot, evals, launches, restarts, life, trace_f = 0, 0.0, 0.0, 0, 0, 0, None, None
    timers_tot = {}
    ctx.timing(True)
    ctx.timing_read(reset=True)
    first = True
    rep_ms = []
    t_loop = time.perf_counter()
    while True:
        run = cg.MinimizerRun(obj, x0, cfg, ls, **qkw)
        ctx.timing(False)
        for _ in range(W):
            assert run.step() is None, f"run ended during warm-up: {run.ret.status}"
        ctx.timing(True)
        ctx.timing_read(reset=True)
        barrier()
        if first:
            sampler.mark_begin()
            first = False
        done, ms = 0, 0.0
        while done < K:
            e0 = torch.cuda.Event(enable_timing=True)
            t0 = t1 = time.perf_counter()
            e0.record(stream)
            e1 = e0
            ended = False
            l0 = l1 = ctx.kernel_launches
            while done < K:
                if run.step() is not None:      # line search at the FP64 floor: that step is not timed
                    ended = True
                    break
                done += 1
                evals += int(run.fdf_evals_ran)
                e1 = torch.cuda.Event(enable_timing=True)
                e1.record(stream)
                t1 = time.perf_counter()
                l1 = ctx.kernel_launches
            torch.cuda.synchronize()
            launches += l1 - l0
            wall_tot += (t1 - t0) * 1e3
            if e1 is not e0:
                ms += e0.elapsed_time(e1)
            if trace_f is None:
                trace_f = run.ret.trace.objective[:max(run.n - 1, 0)].copy()
            if ended and done < K:
                assert run.ret.iters_ran > 0, f"restarted run made no progress: {run.ret.status}"
                life = run.ret.iters_ran if life is None else min(life, run.ret.iters_ran)
                run.info.close()
                run = cg.MinimizerRun(obj, x0, cfg, ls, **qkw)
                restarts += 1
        for k, v in ctx.timing_read(reset=True).items():
            a = timers_tot.setdefault(k, [0.0, 0])
            a[0] += v[0]; a[1] += v[1]
        reps += 1
        # every rank repeats the same number of times: decide on the slowest rank's clock
        tms = torch.tensor([ms], dtype=torch.float64, device="cuda")
        if world > 1:
            import torch.distributed as dist
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        ms_tot += float(tms.item())
        rep_ms.append(float(tms.item()))
        # (the wall-clock guard is rank 0's and every rank applies rank 0's verdict through the reduced flag below)
        stop = ms_tot * 1e-3 >= args.min_timed_s or reps >= args.max_reps or time.perf_counter() - t_loop > 90.0
        tstop = torch.tensor([1.0 if stop else 0.0], dtype=torch.float64, device="cuda")
        if world > 1:
            import torch.distributed as dist
            dist.all_reduce(tstop, op=dist.ReduceOp.MAX)
        if float(tstop.item()) > 0:
            break
        run.info.close()
    sampler.mark_end()
    barrier()
    ctx.timing(False)
    clocks = sampler.stop() if rank == 0 else None
    outputs = run_outputs(run, DUMP_ENTRIES // world) if dump else None
    run.info.close()
    return {"K": K, "W": W, "reps": reps, "ms": ms_tot / reps, "ms_median": float(np.median(rep_ms)),
            "timed_region_s": ms_tot * 1e-3, "wall_ms": wall_tot / reps,
            "evals": evals / reps, "evals_total": evals, "launches": launches / reps, "restarts": restarts, "life": life,
            "trace": trace_f, "timers": {k: (v[0] / reps, v[1] / reps) for k, v in timers_tot.items()}, "clocks": clocks,
            "qkw": qkw, "outputs": outputs}


def roofline_of(args, obj, m, n, coh, world, n_local, nnz_local):
    """dominant-kernel roofline (CUDA events on the launching stream, inside the timed region)"""
    peak, peak_src = peaks()
    timers, evals, K, ms = m["timers"], m["evals"], m["K"], m["ms"]
    dom_per_eval = 2          # launches of the dominant kernel per fdf! (K_b + K_c)
    if args.workload == "rosenbrock":
        dom = "k_blas1<RosenTrial> (fused trial: xp, f, g+, every dot)"
        dom_per_eval = 1
        dom_bytes = algorithmic_bytes(args, n_local, 0, evals, K)      # all bytes are trial-kernel bytes
        dom_ms, dom_cnt = timers["trial"]
    elif args.workload == "logreg":
        dom = ("k_csr_rows (K_b: margins + loss; K_c: g+ = A^T c / N + lambda w + dot pack), one pass per "
               "L2-sized column block of the gathered vector")
        dom_ms = timers["spmv"][0] + timers["spmvT"][0]
        dom_cnt = timers["spmv"][1] + timers["spmvT"][1]
        n_evals = timers["axpy"][1]          # one K_a per fdf!; K_b / K_c may take several column-block passes
        dom_bytes = n_evals * logreg_bytes(args, n_local, nnz_local)[1]
        dom_per_eval = dom_cnt / max(n_evals, 1)
    else:
        direct = obj.trial_site == (2, 4)     # gather-bound matrix: k_spmv_direct, the dots are BLAS-1 passes
        dom = ("k_spmv_direct (K_b: r = A xp - b; K_c: g+ = A^T r; sliced layout, no reductions)" if direct else
               "k_csr_rows (K_b: r = A xp - b; K_c: g+ = A^T r + dot pack)")
        dom_ms = timers["spmv"][0] + timers["spmvT"][0]
        dom_cnt = timers["spmv"][1] + timers["spmvT"][1]
        # per launch pair: 2 x matrix stream + (gather 8n + R b 8n + W r 8n) + (gather 8n + W g+ 8n [+ R u,g 16n fused epilogue])
        dom_bytes = (dom_cnt / 2.0) * (2 * matrix_bytes(n_local, nnz_local) + (40.0 if direct else 56.0) * n_local)
    achieved = dom_bytes / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else 0.0
    traffic, traffic_src = ncu_traffic(args, world, n, coh)
    total_bytes = algorithmic_bytes(args, n_local, nnz_local, evals, K)
    if args.workload == "sparse_ls" and obj.trial_site == (2, 4):
        total_bytes += 16.0 * n_local * evals                          # Σ r² and the eight dots as separate passes
    return {"bound": "hbm", "kernel": dom, "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
            "frac": round(achieved / peak, 4), "traffic": traffic, "traffic_source": traffic_src,
            "algorithmic_bytes_per_launch": round(dom_bytes / max(dom_cnt, 1), 1), "peak_source": peak_src,
            "launches": dom_cnt, "avg_launch_ms": round(dom_ms / max(dom_cnt, 1), 4),
            "frac_of_nominal_8TBs": round(achieved / 8000.0, 4),
            "whole_iteration_GBs_per_gpu": round(total_bytes / (ms * 1e-3) / 1e9, 1),
            "whole_iteration_frac": round(total_bytes / (ms * 1e-3) / 1e9 / peak, 4),
            "kernel_share_of_step": round((dom_ms / max(dom_cnt, 1)) * dom_per_eval * evals / ms, 4),
            "timers_ms": {k: round(v[0], 3) for k, v in timers.items() if v[1]},
            "timers_launches": {k: round(v[1], 1) for k, v in timers.items() if v[1]},
            "fdf_evals_per_s": round(evals / (ms * 1e-3), 2)}


def run_ours(args):
    import torch
    import cgoptim_b200 as cg

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback "
                         "(use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = cg.Context(local_rank)
    if args.gather_block_mib > 0:
        ctx.set_gather_block_bytes(int(args.gather_block_mib * (1 << 20)))
    if args.reduction_ctas:
        ctx.set_reduction_ctas(args.reduction_ctas)
    if world > 1:
        ctx.comm_init_torch()
    n = args.n or FULL_N[args.workload]
    stream = torch.cuda.ExternalStream(ctx.stream_ptr, device=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    obj, x0 = make_objective(cg, args, ctx, n)
    n_local = obj.n_local
    nnz_local = 10 * n_local if args.workload == "sparse_ls" else 0
    if args.workload == "logreg":
        nnz_local = 20 * shard_len(int(n * LOGREG_SAMPLES_PER_FEATURE), world, rank)
    coh = args.coh

    # ---------------- device-resident throughput (`value`) ----------------
    dump = args.dump_outputs is not None
    m = measure_device(cg, torch, args, ctx, obj, x0, n, coh, world, rank, local_rank, stream, barrier, dump)
    outputs = m["outputs"]
    K, W, ms, qkw, life = m["K"], m["W"], m["ms"], m["qkw"], m["life"]
    roofline = roofline_of(args, obj, m, n, coh, world, n_local, nnz_local)
    par, par_note = parity_vs_n1(args, n, coh, m["trace"])
    if rank == 0:
        parity_gate(args, par, f"{args.workload} n={n} coh_log2={coh}")

    # ---------------- end-to-end through the public API (`e2e`) ----------------
    e2e = None
    if not args.no_e2e:
        x0p = torch.from_numpy(x0.copy()).pin_memory().numpy()

        def public_call(kw):
            """K iterations through `minimizeobjective` with host vectors -> (seconds, max over ranks; evals; calls)"""
            # one untimed call first: page-locks the result buffers (they are pooled and reused) and
            # warms the allocator, as a long-running host would have done
            cfg1, ls1 = solver_configs(cg, 1, args.workload)
            cg.minimizeobjective(obj, x0p, cfg1, ls1, **kw)
            remaining, dt, ev2, calls = K, 0.0, 0, 0
            while remaining > 0:                                 # more than one call only if a run hits the FP64 floor
                per_call = remaining if life is None else max(1, min(remaining, life - 3))
                cfg2, ls2 = solver_configs(cg, per_call, args.workload)
                barrier()
                t0 = time.perf_counter()
                ret = cg.minimizeobjective(obj, x0p, cfg2, ls2, **kw)  # H2D x0 … iterations … D2H x, g
                barrier()
                dt += time.perf_counter() - t0
                assert ret.iters_ran > 0, (ret.iters_ran, ret.status)
                remaining -= ret.iters_ran
                ev2 += int(ret.trace.objective_evals.sum())
                calls += 1
            tdt = torch.tensor([dt], dtype=torch.float64, device="cuda")
            if world > 1:
                import torch.distributed as dist
                dist.all_reduce(tdt, op=dist.ReduceOp.MAX)
            return float(tdt.item()), ev2, calls

        dt, ev2, calls = public_call(qkw)
        e2e = {"value": round(K / dt, 4), "unit": "iterations/s",
               "h2d_bytes_per_step": round((8.0 * n_local * calls + 16.0 * (ev2 + K)) / K, 1),
               "d2h_bytes_per_step": round((16.0 * n_local * calls + 128.0 * (ev2 + 2 * K)) / K, 1),
               "api_calls": calls,
               "includes": "x0 H2D from pinned host memory, f/g at x0, K iterations (scalar pack D2H "
                           "every launch), minimizer+gradient D2H", "wall_s": round(dt, 4)}
        if args.workload == "sparse_ls" and not qkw:
            # the same call with the quadratic-aware line search (SURVEY.md §8f N1: one SpMV + one SpMVᵀ per iteration
            # whatever the number of trials — the first line search of a run takes five): reported beside the
            # headline, which stays the plain path
            try:            # (line-search scalars are replicated, so every rank takes the same branch here)
                dtq, evq, callsq = public_call({"quadratic_linesearch": True})
                e2e["quadratic_aware_linesearch"] = {"value": round(K / dtq, 4), "unit": "iterations/s",
                                                     "api_calls": callsq, "fdf_evals": evq, "wall_s": round(dtq, 4)}
            except AssertionError as e:
                e2e["quadratic_aware_linesearch"] = {"error": str(e)[:200]}

    # ---------------- the other matrix variant of cfg 3, same run (`secondary`) ----------------
    secondary = None
    if args.workload == "sparse_ls" and not args.no_secondary:
        coh2 = 30 if coh < 28 else 0
        obj.close()
        del obj
        args2 = argparse.Namespace(**vars(args))
        args2.coh = coh2
        obj2, x02 = make_objective(cg, args2, ctx, n)
        m2 = measure_device(cg, torch, args2, ctx, obj2, x02, n, coh2, world, rank, local_rank, stream, barrier, dump)
        if dump:
            outputs.update({"secondary_" + k: v for k, v in m2["outputs"].items()})
        r2 = roofline_of(args2, obj2, m2, n, coh2, world, n_local, nnz_local)
        p2, p2_note = parity_vs_n1(args2, n, coh2, m2["trace"])
        secondary = {("coh%d" % coh2): {
            "workload": workload_text(args2, n, coh2), "value": round(m2["K"] / (m2["ms"] * 1e-3), 4), "unit": "iterations/s",
            "ms_per_step": round(m2["ms"] / m2["K"], 4), "repetitions": m2["reps"], "timed_region_s": round(m2["timed_region_s"], 3),
            "ms_per_step_median_over_repetitions": round(m2["ms_median"] / m2["K"], 4),
            "fdf_evals_per_repetition": m2["evals"], "roofline": r2, "clocks": m2["clocks"],
            "parity_vs_n1": p2, "parity_vs_n1_note": p2_note,
            "objective_trace_head": [float(v) for v in m2["trace"][:4]]}}
        if args.write_fixture and world == 1:
            write_fixture(args2, n, coh2, m2["trace"])
        obj2.close()
    if args.write_fixture and world == 1:
        write_fixture(args, n, coh, m["trace"])
    if dump:
        write_outputs(args.dump_outputs, outputs, rank, world)

    line = None
    if rank == 0:
        line = {
            "metric": "lbfgs_iterations_per_s" if args.workload == "logreg" else "cg_iterations_per_s",
            "value": round(K / (ms * 1e-3), 4), "unit": "iterations/s",
            "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": round(ms / K, 4),
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": workload_text(args, n, coh),
                       "n": n, "sharding": f"rows/vector slices over {world} rank(s)",
                       "l2_policy": "inputs larger than L2 (vectors are 8n bytes >> 126 MB)",
                       "repetitions": m["reps"], "timed_region_s": round(m["timed_region_s"], 3),
                       "ms_per_step_median_over_repetitions": round(m["ms_median"] / K, 4),
                       "fdf_evals_in_timed_region": m["evals_total"], "restarts_in_timed_region": m["restarts"],
                       "quadratic_aware_linesearch": bool(qkw), "host": "python/ctypes over the C ABI",
                       "value_is": ("coh_log2=%d; the other matrix variant of cfg 3 is under `secondary`" % coh)
                       if args.workload == "sparse_ls" else "the only variant"},
            "roofline": roofline, "e2e": e2e, "gpu_launches": int(round(m["launches"])), "clocks": m["clocks"],
            "host_wall_ms_per_step": round(m["wall_ms"] / K, 4),
            "parity_vs_n1": par, "parity_vs_n1_note": par_note, "parity_tol": PARITY_TOL,
            "objective_trace_head": [float(v) for v in m["trace"][:4]],
            "secondary": secondary,
        }
    return line, ctx


def write_fixture(args, n, coh, trace):
    try:
        with open(FIXTURE) as f:
            data = json.load(f)
    except (OSError, ValueError):
        data = {"generator": "python bench.py --gpus 1 --write-fixture (on a B200)", "traces": {}}
    data["traces"][fixture_key(args, n, coh)] = [float(v).hex() for v in trace]
    os.makedirs(os.path.dirname(FIXTURE), exist_ok=True)
    with open(FIXTURE, "w") as f:
        json.dump(data, f, indent=0)


# ------------------------------------------------------------------------------ batched (cfg 5)
def run_batched(args):
    """BASELINE.json configs[4]: 262,144 independent n = 512 Rosenbrock problems, HZ + strong Wolfe,
    one CTA per problem, problems split over the ranks without communication ("weak" per problem;
    total work fixed).  A step = one whole batched solve of this rank's share."""
    import torch
    import cgoptim_b200 as cg
    from oracle import oracle as O

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = cg.Context(local_rank)
    n = args.n or 512
    nprob = BATCHED_NPROB // world
    rng = np.random.default_rng(24 + rank)
    X0 = np.tile([-1.2, 1.0], n // 2)[None, :] + 0.1 * (2.0 * rng.random((nprob, n)) - 1.0)
    X0p = torch.from_numpy(X0).pin_memory().numpy()
    cfg = cg.setupCGConfig(1e-5, cg.HagerZhang(), cg.DisableTrace(), max_iters=1000)
    ls = cg.setupStrongWolfeBisection(1e-5, 0.8, a_max_growth_factor=2.0, max_iters=1000, zoom_max_iters=100)
    K, W = max(args.steps, 1), max(min(args.warmup, 3), 1)
    for _ in range(W):
        res = cg.minimizeobjective_batched(X0p, cfg, ls, ctx)
    ctx.timing(True)
    ctx.timing_read(reset=True)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = ctx.kernel_launches
    torch.cuda.synchronize()
    sampler.mark_begin()
    t0 = time.perf_counter()
    for _ in range(K):
        res = cg.minimizeobjective_batched(X0p, cfg, ls, ctx)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    sampler.mark_end()
    clocks = sampler.stop() if rank == 0 else None
    kms = ctx.timing_read(reset=True)["batched"][0]
    ctx.timing(False)
    if args.dump_outputs is not None:          # the last solve's per-problem results, the minimizers of sampled problems
        rows = sample_index(nprob, max(DUMP_ENTRIES // (world * n), 1))
        write_outputs(args.dump_outputs, {
            "minimizer": res.minimizer[rows], "sample_index": rows, "objective": res.objective,
            "grad_norm": res.grad_norm, "iters_ran": res.iters_ran, "status_code": res.status_code,
            "fdf_evals": res.fdf_evals}, rank, world)
    t = torch.tensor([kms, wall], dtype=torch.float64, device="cuda")
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    kms, wall = float(t[0].item()), float(t[1].item())
    iters = torch.tensor([float(res.iters_ran.sum()), float(res.fdf_evals.sum()),
                          float((res.status_code == 1).sum())], dtype=torch.float64, device="cuda")
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(iters)
    tot_it, tot_ev, tot_ok = (float(v) for v in iters.tolist())
    line = None
    if rank == 0:
        line = {"metric": "batched_cg_iterations_per_s", "value": round(tot_it * K / (kms * 1e-3), 1),
                "unit": "iterations/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": round(kms / K, 3),
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": f"{BATCHED_NPROB} independent extended-Rosenbrock problems n={n}, Hager-Zhang CG + "
                                       f"StrongWolfeBisection(1e-5,0.8), eps 1e-5, one CTA per problem, whole solver on device",
                           "problems_per_s": round(nprob * world * K / (kms * 1e-3), 1),
                           "iterations_total": tot_it, "fdf_evals_total": tot_ev, "converged": tot_ok,
                           "l2_policy": "on-chip workload: x0 read once, result written once (HBM roofline not applicable)"},
                # FP64 instructions the kernel issues per element pair and trial (Hager-Zhang: x + a u 4, objective and
                # gradient 12, y 2, six dots 25); no FMA anywhere (the reference's arithmetic is unfused), so the
                # pipe's ceiling is one DADD/DMUL per FP64 lane and clock: 64 lanes x SMs x max SM clock
                "roofline": {"bound": "fp64 pipe (on-chip: registers + shuffles; HBM roofline not applicable)",
                             "achieved": round(tot_ev * K * (n / 2) * 43 / (kms * 1e-3) / 1e12 / world, 3),   # per GPU, like the peak
                             "peak": round(64 * ctx.sm_count * (clocks or {}).get("sm_max_mhz", 1965.0) * 1e6 / 1e12, 3)
                             if clocks and clocks.get("sm_max_mhz") else round(64 * ctx.sm_count * 1965e6 / 1e12, 3),
                             "unit": "TFLOP/s per GPU (unfused FP64 instructions)", "frac": None, "traffic": None,
                             "peak_source": "nominal: 64 FP64 lanes/SM/clk x SM count x max SM clock, FMA not usable"},
                "e2e": {"value": round(tot_it * K / wall, 1), "unit": "iterations/s",
                        "h2d_bytes_per_step": 8.0 * nprob * n, "d2h_bytes_per_step": 8.0 * nprob * n + 36.0 * nprob,
                        "includes": "x0 H2D from pinned memory, solve, minimizers + per-problem results D2H"},
                "gpu_launches": int(ctx.kernel_launches - l0), "clocks": clocks, "cpu_baseline": None}
    if line is not None and line["roofline"]["peak"]:
        line["roofline"]["frac"] = round(line["roofline"]["achieved"] / line["roofline"]["peak"], 4)
    return line, ctx


# ------------------------------------------------------------------------------ CPU arm
CPU_ITERS = 10          # iterations the CPU arm times (both in the main line's cpu_baseline and in --impl reference)


def run_cpu(args, steps, warmup, threads):
    """The reference's CPU path on the host cores (BASELINE.md §3): the oracle's C restatement in the reference's
    own shape — unfused passes, allocating getβ, sequential sums (src/cg_utils.jl:13-20, src/cg_flavours.jl:96-105,
    src/engine/optim.jl:136-140) — at n/10 of the full size with linear extrapolation (flagged), in two rows:
    1 thread (Julia's own loops are single-threaded) and all cores (OpenMP on fdf! and dot/norm, emulating a
    threaded OpenBLAS).  The same `steps` in the main line's cpu_baseline and in the --impl reference arm."""
    from oracle import oracle as O
    n_full = args.n or FULL_N[args.workload]
    n = min(SAMPLE_N[args.workload], n_full)
    if args.workload == "rosenbrock":
        obj = O.Objective.rosenbrock(n)
        x0 = O.rosenbrock_x0(n, 24, 0.1)
    elif args.workload == "logreg":
        obj = O.Objective.logreg(int(n * LOGREG_SAMPLES_PER_FEATURE), n, 20, 24, 1e-6, threads)
        x0 = np.zeros(n)
    else:
        obj = O.Objective.sparse_ls(n, 10, min(1 << 20, (n - 1) // 2), 24, args.coh, threads)
        x0 = np.zeros(n)

    def mk(it, th):
        if args.workload == "logreg":
            return O.make_config("LBFGS", "StrongWolfeBisection", eps=1e-300, max_iters=it, lbfgs_m=10,
                                 c1=1e-4, c2=0.9, sum_mode="seq", threads=th)
        return O.make_config("HagerZhang", "StrongWolfeBisection", eps=1e-300, max_iters=it,
                             sum_mode="seq", beta_form="literal", threads=th)

    rows = []
    for th, its in ((threads, steps), (1, max(2, steps // 3))):
        if th == 1 and threads == 1 and rows:
            break
        obj.set_sum_mode("seq", th)
        if warmup and th == threads:
            O.minimize(obj, x0, mk(warmup, th), trace=False)
        t0 = time.perf_counter()
        r = O.minimize(obj, x0, mk(its, th))       # one fdf! at x0 is inside the timed call, as in minimizeobjective
        dt = time.perf_counter() - t0
        rows.append({"threads": th, "iterations": int(r.iters_ran), "seconds": round(dt, 3),
                     "sample_iterations_per_s": r.iters_ran / dt, "value": r.iters_ran / dt * (n / n_full)})
    best = rows[0]
    return {"value": best["value"], "unit": "iterations/s", "cores": threads, "kind": "port",
            "sample": (f"oracle C restatement of the reference (Julia not installed: 'julia thread count' n/a), "
                       f"reference-shaped arithmetic, {best['iterations']} iterations at n={n} (= n_full/{n_full // n}, "
                       f"BASELINE.md §3) in {best['seconds']:.2f}s = {best['sample_iterations_per_s']:.3f} it/s, "
                       f"scaled linearly by n/n_full = {n}/{n_full}; OpenMP threads on fdf! and dot/norm = {threads}; "
                       f"1-thread row: {rows[-1]['value']:.5f} it/s"),
            "sample_n": n, "extrapolated": n != n_full, "sample_iterations_per_s": best["sample_iterations_per_s"],
            "single_thread": rows[-1] if rows[-1]["threads"] == 1 else None, "rows": rows, "host_cores": os.cpu_count()}


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    if args.impl == "reference":
        if args.dump_outputs is not None:
            raise SystemExit("bench.py: --dump-outputs writes the outputs of the device path (--impl ours)")
        if rank != 0:
            return
        threads = os.cpu_count() or 1
        cb = run_cpu(args, CPU_ITERS, 0, threads)
        n = args.n or FULL_N[args.workload]
        line = {"impl": "reference", "metric": "lbfgs_iterations_per_s" if args.workload == "logreg" else "cg_iterations_per_s", "value": round(cb["value"], 6),
                "unit": "iterations/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": round(1e3 / cb["value"], 3), "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": workload_text(args, n, args.coh), "n": n, "sample_n": cb["sample_n"],
                           "cpu_iterations_timed": CPU_ITERS, "extrapolated_from_sample": cb["extrapolated"]},
                "cpu_baseline": cb,
                "e2e": {"value": round(cb["value"], 6), "unit": "iterations/s", "h2d_bytes_per_step": 0,
                        "d2h_bytes_per_step": 0}}
        print(json.dumps(line), flush=True)
        return
    line, ctx = run_batched(args) if args.workload == "batched" else run_ours(args)
    if rank == 0:
        world = int(os.environ.get("WORLD_SIZE", "1"))
        if world == 1 and not args.no_cpu_baseline and args.workload != "batched":
            line["cpu_baseline"] = run_cpu(args, CPU_ITERS, 0, os.cpu_count() or 1)
        else:
            line["cpu_baseline"] = None
        print(json.dumps(line), flush=True)
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
        # peer-mapped device memory and two NCCL communicators are still open: leave their
        # teardown to process exit instead of the interpreter's unordered finalisers
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
