"""Evaluation rates of logistic regression on a host CSR (LogRegGPU_from_csr) on one GPU.

  (a) parity: N = d = 1e7, K = 20 (2e8 entries, column-blocked on both sides), the synthetic LogRegGPU against
      LogRegGPU_from_csr on its downloaded CSR and labels, alternated three times;
  (b) the cliff and its fix: the same matrix plus a ones column (the intercept: a row of Aᵀ with N entries), on the
      default path (long-row kernels) and forced onto k_csr_rows (CGO_CSR_MODE = 1: that row on one lane), against
      the matrix without the column;
  (c) the threshold: K_c (the SpMVᵀ class) for one row of ℓ = 2^8 … 2^24 entries on k_spmv_direct, split into work
      units against summed on one lane.  The one-lane arm runs a build of the library with CGO_LONG_ROW raised above
      every ℓ (--seq-lib), in a child process.

Rates are evaluations per second of cgo_eval_trial after warm-up: the host clock around calls that end in a device
synchronise, and the per-class kernel times of the ctx's CUDA-event timing.  Writes profiles/r3_logreg_csr_rates.txt
(or --out) and prints the card name and power limit."""
import argparse
import json
import os
import re
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def long_row_limit():
    with open(os.path.join(ROOT, "include", "cgoptim.h")) as f:
        return int(re.search(r"#define\s+CGO_LONG_ROW\s+(\d+)", f.read()).group(1))


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


def synthetic_csr(cg, ctx, N, d, K):
    ctx.set_gather_block_bytes(0)
    flat = cg.LogRegGPU(N, d, K, 24, 1e-6, ctx)                  # single-pass copy: downloadable at every size
    ctx.set_gather_block_bytes(40 << 20)
    out = flat.csr(False)
    flat.close()
    return out


def with_ones_column(rp, ci, va, d):
    rp1 = rp + np.arange(rp.size, dtype=np.int64)
    ci1 = np.empty(rp1[-1], dtype=np.int32)
    va1 = np.empty(rp1[-1])
    last = rp1[1:] - 1
    mask = np.ones(rp1[-1], dtype=bool)
    mask[last] = False
    ci1[mask], va1[mask] = ci, va
    ci1[last], va1[last] = d, 1.0
    return rp1, ci1, va1


def threshold_arm(lengths, evals):
    """K_c of one row of ℓ entries (ℓ samples whose only feature is the ones column), k_spmv_direct family"""
    import cgoptim_b200 as cg
    ctx = cg.Context(0)
    ctx.timing(True)
    ctx.set_csr_mode(2)
    out = {}
    rng = np.random.default_rng(0)
    for ell in lengths:
        y = np.where(rng.random(ell) < 0.5, -1.0, 1.0)
        obj = cg.LogRegGPU_from_csr(ell, 1, np.arange(ell + 1, dtype=np.int64), np.zeros(ell, np.int32), np.ones(ell), y,
                                    1e-6, ctx)
        r = rate(obj, ctx, evals)
        out[ell] = r["kernel_ms_per_eval"].get("spmvT", 0.0)
        obj.close()
    ctx.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_logreg_csr_rates.txt"))
    ap.add_argument("--seq-lib", default=None, help="libcgoptim.so built with CGO_LONG_ROW above 2^24")
    ap.add_argument("--skip-large", action="store_true")
    a = ap.parse_args()
    lengths = [1 << k for k in range(8, 25)]
    import cgoptim_b200 as cg
    props = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True).stdout.strip()
    lines = [f"# logistic regression on a host CSR, one GPU: {props}", f"# CGO_LONG_ROW = {long_row_limit()}"]
    print(lines[0], flush=True)
    ctx = cg.Context(0)
    ctx.timing(True)
    if not a.skip_large:
        N = d = 10_000_000
        rp, ci, va, y = synthetic_csr(cg, ctx, N, d, 20)
        syn = cg.LogRegGPU(N, d, 20, 24, 1e-6, ctx)
        usr = cg.LogRegGPU_from_csr(N, d, rp, ci, va, y, 1e-6, ctx)
        lines.append(f"(a) parity N = d = 1e7, K = 20: blocks A {syn.csr_blocks(False)} / {usr.csr_blocks(False)}, "
                     f"Aᵀ {syn.csr_blocks(True)} / {usr.csr_blocks(True)}")
        for rep in range(3):
            for name, o in (("LogRegGPU", syn), ("LogRegGPU_from_csr", usr)):
                r = rate(o, ctx, 20)
                lines.append(f"    rep {rep} {name:20s} {r['evals_per_s']:8.2f} evals/s  {r['ms_per_eval']:8.3f} ms  "
                             f"kernels {json.dumps({k: round(v, 3) for k, v in r['kernel_ms_per_eval'].items()})}")
                print(lines[-1], flush=True)
        syn.close()
        base = rate(usr, ctx, 20)
        usr.close()
        rp1, ci1, va1 = with_ones_column(rp, ci, va, d)
        del rp, ci, va
        lines.append("(b) the same matrix plus a ones column (Aᵀ gains a row of 1e7 entries)")
        lines.append(f"    without the column, default path  {base['evals_per_s']:8.2f} evals/s  {base['ms_per_eval']:9.3f} ms  "
                     f"kernels {json.dumps({k: round(v, 3) for k, v in base['kernel_ms_per_eval'].items()})}")
        for mode, ev in ((0, 20), (1, 2)):
            ctx.set_csr_mode(mode)
            one = cg.LogRegGPU_from_csr(N, d + 1, rp1, ci1, va1, y, 1e-6, ctx)
            r = rate(one, ctx, ev, warm=1)
            lines.append(f"    with the column, mode {mode} ({'long-row kernels' if mode == 0 else 'k_csr_rows, one lane'})"
                         f"  {r['evals_per_s']:8.2f} evals/s  {r['ms_per_eval']:9.3f} ms  "
                         f"kernels {json.dumps({k: round(v, 3) for k, v in r['kernel_ms_per_eval'].items()})}")
            print(lines[-1], flush=True)
            one.close()
        ctx.set_csr_mode(0)
        del rp1, ci1, va1
    ctx.close()
    split = threshold_arm(lengths, 20)
    seq = {}
    if a.seq_lib:
        res = subprocess.run([sys.executable, "-c",
                              "import sys, json; sys.path.insert(0, %r); import cgoptim_b200 as cg; "
                              "from cgoptim_b200 import _capi; _capi.LIB_PATH = %r; "
                              "sys.path.insert(0, %r); import logreg_csr_rates as m; "
                              "print('JSON', json.dumps(m.threshold_arm(%r, 5)))"
                              % (ROOT, os.path.abspath(a.seq_lib), os.path.join(ROOT, "profiles"), lengths)],
                             capture_output=True, text=True)
        for ln in res.stdout.splitlines():
            if ln.startswith("JSON "):
                seq = {int(k): v for k, v in json.loads(ln[5:]).items()}
        if not seq:
            print(res.stdout[-2000:], res.stderr[-4000:])
    lines.append("(c) K_c (spmvT class, ms per evaluation) of one row of ℓ entries on k_spmv_direct: work units vs one lane")
    lines.append(f"    {'ℓ':>10s} {'split':>10s} {'one lane':>10s}")
    for ell in lengths:
        lines.append(f"    {ell:10d} {split[ell]:10.4f} {seq.get(ell, float('nan')):10.4f}")
    with open(a.out, "w") as f:
        f.write("\n".join(lines) + "\n")
    print("\n".join(lines))


if __name__ == "__main__":
    main()
