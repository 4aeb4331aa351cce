"""Evaluation rates of softmax regression on a host CSR (SoftmaxRegGPU_from_csr) on one GPU.

  (a) N = 1e7 samples, d = 1e6 features, 20 random features per sample plus an intercept (2.1e8 entries), K = 4, 10,
      32: evaluations per second and the per-class kernel times of a trial (spmv = K_b, the SpMM of A and the
      long rows; spmvT = K_c, the SpMM of Aᵀ and the intercept's long row; other = softmax and /N + λW).  The binary
      LogRegGPU_from_csr on the same matrix and labels mod 2 is recorded for scale.
  (b) the path that needs no new kernel: the same SpMVs done by k_spmv_direct on the Kronecker-expanded matrix
      A ⊗ I_K (SparseLSGPU_from_csr in CGO_CSR_MODE = 2, its K_b / K_c class times), against the K-column SpMM on
      the same matrix.  The expanded matrix is built on the host, so this arm runs without the intercept (least
      squares keeps sequential sums on long rows) and at 8e8 expanded entries: N = 8e8 / (20 K).

Rates are evaluations per second of cgo_eval_trial after warm-up: the host clock around calls that end in a device
synchronise, and the per-class kernel times of the ctx's CUDA-event timing.  Writes profiles/r3_softmax_csr_rates.txt
(or --out) with the card name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


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
    return {"evals_per_s": 1.0 / wall, "ms_per_eval": 1e3 * wall, "kernel_ms_per_eval": cls}


def fmt(r):
    return (f"{r['evals_per_s']:8.2f} evals/s  {r['ms_per_eval']:9.3f} ms  "
            f"kernels {json.dumps({k: round(v, 3) for k, v in r['kernel_ms_per_eval'].items()})}")


def matrix(N, d, per_row, intercept, seed=5):
    """per_row random features of [0, d − 1) per sample (sorted), then the ones column d − 1 if intercept"""
    rng = np.random.default_rng(seed)
    cols = np.sort(rng.integers(0, d - 1, (N, per_row), dtype=np.int32), axis=1)
    w = per_row + (1 if intercept else 0)
    col = np.empty((N, w), dtype=np.int32)
    col[:, :per_row] = cols
    val = rng.uniform(-1.0, 1.0, (N, w))
    if intercept:
        col[:, per_row] = d - 1
        val[:, per_row] = 1.0
    return np.arange(N + 1, dtype=np.int64) * w, col.ravel(), val.ravel()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_softmax_csr_rates.txt"))
    ap.add_argument("--classes", default="4,10,32")
    ap.add_argument("--evals", type=int, default=10)
    a = ap.parse_args()
    import cgoptim_b200 as cg
    from softmax_csr_reference import kron_csr
    props = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True).stdout.strip()
    lines = [f"# softmax regression on a host CSR, one GPU: {props}"]
    print(lines[0], flush=True)
    classes = [int(k) for k in a.classes.split(",")]
    ctx = cg.Context(0)
    ctx.timing(True)
    N, d = 10_000_000, 1_000_000
    rp, ci, va = matrix(N, d, 20, True)
    y = np.random.default_rng(6).integers(0, 1 << 30, N)
    lines.append(f"(a) N = 1e7, d = 1e6, 20 features per sample + intercept ({rp[-1]} entries)")
    lr = cg.LogRegGPU_from_csr(N, d, rp, ci, va, np.where(y % 2 == 1, 1.0, -1.0), 1e-6, ctx)
    lines.append(f"    binary LogRegGPU_from_csr      blocks A {lr.csr_blocks(False)}, Aᵀ {lr.csr_blocks(True)}  {fmt(rate(lr, ctx, a.evals))}")
    print(lines[-1], flush=True)
    lr.close()
    for K in classes:
        obj = cg.SoftmaxRegGPU_from_csr(N, d, K, rp, ci, va, y % K, 1e-6, ctx)
        lines.append(f"    softmax K = {K:2d}  blocks A {obj.csr_blocks(False):3d}, Aᵀ {obj.csr_blocks(True):3d}  "
                     f"{fmt(rate(obj, ctx, a.evals))}")
        print(lines[-1], flush=True)
        obj.close()
    del rp, ci, va
    lines.append("(b) K-column SpMM against k_spmv_direct on A ⊗ I_K (no intercept, 20 features per sample, 8e8 expanded "
                 "entries; spmv = K_b, spmvT = K_c, ms per evaluation)")
    for K in classes:
        Nc = 800_000_000 // (20 * K)
        rp, ci, va = matrix(Nc, d, 20, False, seed=7)
        yk = np.random.default_rng(8).integers(0, K, Nc)
        obj = cg.SoftmaxRegGPU_from_csr(Nc, d, K, rp, ci, va, yk, 1e-6, ctx)
        rs = rate(obj, ctx, a.evals)
        obj.close()
        erp, eci, eva = kron_csr(Nc, rp, ci, va, K)
        del rp, ci, va
        eci = eci.astype(np.int32)
        ctx.set_csr_mode(2)
        ls = cg.SparseLSGPU_from_csr(Nc * K, d * K, erp, eci, eva, np.zeros(Nc * K), ctx)
        ctx.set_csr_mode(0)
        del erp, eci, eva
        rl = rate(ls, ctx, a.evals)
        ls.close()
        ks, kl = rs["kernel_ms_per_eval"], rl["kernel_ms_per_eval"]
        lines.append(f"    K = {K:2d}, N = {Nc:9d}:  SpMM  K_b {ks.get('spmv', 0.0):8.3f}  K_c {ks.get('spmvT', 0.0):8.3f}   "
                     f"expanded k_spmv_direct  K_b {kl.get('spmv', 0.0):8.3f}  K_c {kl.get('spmvT', 0.0):8.3f}")
        print(lines[-1], flush=True)
    ctx.close()
    with open(a.out, "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
