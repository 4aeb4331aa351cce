"""Evaluation rates of per-sample weights and the unpenalised intercept (LogRegGPU_from_csr / SoftmaxRegGPU_from_csr with
sample_weight and fit_intercept) on one GPU.

N = 1e7 samples, d = 1e6 features, 20 random features per sample; binary and K = 4, 10.  For each objective, in one
run and alternated (each arm measured `--reps` times, round robin):
  ones      an explicit ones column appended as feature d (2.1e8 entries; λ penalises its weight)
  icpt      fit_intercept=True on the same data without the column (2e8 entries): the intercept is the unit row
  icpt+w1   fit_intercept=True with all-ones sample_weight: what reading the weights costs over sample_weight=None
Each line: evaluations per second of cgo_eval_trial after warm-up (the host clock around calls that end in a device
synchronise) and the per-class kernel times of the ctx's CUDA-event timing (spmv = K_b: A and its long rows;
spmvT = K_c: Aᵀ, its long rows and the unit row; other = the loss op and the combine pass).  Writes
profiles/r3_glm_csr_rates.txt (or --out) with the card name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def rate(obj, ctx, evals, warm=2):
    ws = obj.make_workspace(np.zeros(obj.n_local), fuse_direction=False)
    ws.reset_direction()
    for _ in range(warm):
        ws.eval_trial(1e-3)
    ctx.timing_read(reset=True)
    t0 = time.perf_counter()
    for _ in range(evals):
        ws.eval_trial(1e-3)
    wall = (time.perf_counter() - t0) / evals
    cls = {k: ms / evals for k, (ms, c) in ctx.timing_read(reset=True).items() if c}
    ws.close()
    return {"evals_per_s": 1.0 / wall, "kernel_ms_per_eval": cls}


def fmt(r):
    return (f"{r['evals_per_s']:8.2f} evals/s  "
            f"kernels {json.dumps({k: round(v, 3) for k, v in r['kernel_ms_per_eval'].items()})}")


def matrix(N, d, per_row, ones, seed=5):
    """per_row random features of [0, d) per sample (sorted), then the ones column d if `ones`"""
    rng = np.random.default_rng(seed)
    cols = np.sort(rng.integers(0, d, (N, per_row), dtype=np.int32), axis=1)
    w = per_row + (1 if ones else 0)
    col = np.empty((N, w), dtype=np.int32)
    col[:, :per_row] = cols
    val = rng.uniform(-1.0, 1.0, (N, w))
    if ones:
        col[:, per_row] = d
        val[:, per_row] = 1.0
    return np.arange(N + 1, dtype=np.int64) * w, col.ravel(), val.ravel()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_glm_csr_rates.txt"))
    ap.add_argument("--classes", default="1,4,10", help="1 = binary")
    ap.add_argument("--evals", type=int, default=10)
    ap.add_argument("--reps", type=int, default=2)
    a = ap.parse_args()
    import cgoptim_b200 as cg
    props = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True).stdout.strip()
    lines = [f"# logistic / softmax regression with weights and an intercept, one GPU: {props}"]
    print(lines[0], flush=True)
    ctx = cg.Context(0)
    ctx.timing(True)
    N, d = 10_000_000, 1_000_000
    rp1, ci1, va1 = matrix(N, d, 20, True)
    rp0, ci0, va0 = matrix(N, d, 20, False)
    y = np.random.default_rng(6).integers(0, 1 << 30, N)
    ones = np.ones(N)
    lines.append(f"N = 1e7, d = 1e6, 20 features per sample; ones column: {rp1[-1]} entries, without: {rp0[-1]}")
    for K in [int(k) for k in a.classes.split(",")]:
        def make(arm):
            rp, ci, va, nf = (rp1, ci1, va1, d + 1) if arm == "ones" else (rp0, ci0, va0, d)
            sw = ones if arm == "icpt+w1" else None
            icpt = arm != "ones"
            if K == 1:
                return cg.LogRegGPU_from_csr(N, nf, rp, ci, va, np.where(y % 2 == 1, 1.0, -1.0), 1e-6, ctx,
                                             sample_weight=sw, fit_intercept=icpt)
            return cg.SoftmaxRegGPU_from_csr(N, nf, K, rp, ci, va, y % K, 1e-6, ctx, sample_weight=sw,
                                             fit_intercept=icpt)
        name = "binary" if K == 1 else f"softmax K = {K}"
        for rep in range(a.reps):
            for arm in ("ones", "icpt", "icpt+w1"):
                obj = make(arm)
                lines.append(f"    {name:14s} {arm:8s} rep {rep}  blocks A {obj.csr_blocks(False)}, Aᵀ "
                             f"{obj.csr_blocks(True):2d}  bytes/eval {obj.bytes_per_eval:.4e}  {fmt(rate(obj, ctx, a.evals))}")
                print(lines[-1], flush=True)
                obj.close()
    ctx.close()
    with open(a.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
