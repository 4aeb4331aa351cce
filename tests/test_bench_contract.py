"""CPU checks of bench.py: the byte-accounting helpers behind `roofline.achieved`, the shard helper, the
ncu-traffic lookup, the reference arm's JSON line (the one leg of bench.py that runs without a GPU) and the
files of --dump-outputs; on the GPU, that --steps K times K steps and two runs dump the same outputs."""
import importlib.util
import json
import os
import subprocess
import sys
import types

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def bench():
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _args(**kw):
    a = types.SimpleNamespace(workload="sparse_ls", coh=30, n=0)
    a.__dict__.update(kw)
    return a


def test_algorithmic_bytes_formulas(bench):
    n, nnz = 200_000_000, 2_000_000_000
    M = 12.0 * nnz + 8.0 * (n + 1)
    assert bench.matrix_bytes(n, nnz) == M
    # DESIGN.md §5: CSR-LS E(2M + 80n) + 16n per iteration; Rosenbrock 8n(6 + 5(E − 1))
    assert bench.algorithmic_bytes(_args(), n, nnz, evals=3, iters=2) == 3 * (2 * M + 80.0 * n) + 2 * 16.0 * n
    assert bench.algorithmic_bytes(_args(workload="rosenbrock"), n, 0, evals=5, iters=3) == 8.0 * n * (6 * 3 + 5 * 2)


def test_shard_len_matches_the_c_abi(bench):
    import cgoptim_b200 as cg
    for n, world in ((200_000_000, 8), (50_000_000, 3), (2002, 2)):
        for r in range(world):
            lo, hi = cg.shard_range(n, world, r, 2)
            assert bench.shard_len(n, world, r) == hi - lo


def test_ncu_traffic_lookup(bench):
    t, src = bench.ncu_traffic(_args(), 1, 200_000_000)
    assert t is not None and abs(t - 31.2e9) < 0.1e9 and "r1_ncu_full_ls_r1b.txt" in src
    assert bench.ncu_traffic(_args(), 2, 200_000_000) == (None, None)          # other configuration: no number
    t0, src0 = bench.ncu_traffic(_args(coh=0), 1, 200_000_000)                # the banded-random headline: r2 capture
    assert t0 is not None and abs(t0 - 30.5e9) < 0.3e9 and "k_spmv_direct" in src0
    assert bench.ncu_traffic(_args(coh=5), 1, 200_000_000) == (None, None)
    assert bench.ncu_traffic(_args(workload="logreg"), 1, 20_000_000) == (None, None)


def test_reference_arm_line():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                        "--warmup", "0", "--n", "400000"], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0, p.stderr[-2000:]
    d = json.loads(p.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "iterations/s" and d["value"] > 0 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == pytest.approx(d["value"], rel=1e-4)
    assert d["e2e"] == {"value": d["value"], "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # BASELINE.md §3: a 1-thread row beside the all-core one, both on the same sample
    cb = d["cpu_baseline"]
    assert cb["rows"][0]["threads"] == cb["cores"] and cb["rows"][0]["iterations"] == 10
    assert cb["single_thread"] is None or cb["single_thread"]["threads"] == 1
    assert d["config"]["n"] == 400000 and "coh_log2=0" in d["config"]["workload"]


def test_parity_fixture_lookup(bench, tmp_path, monkeypatch):
    import numpy as np
    monkeypatch.setattr(bench, "FIXTURE", str(tmp_path / "fx.json"))
    a = _args(coh=0, quadratic_ls=False)
    tr = np.array([3.0, 2.0, 1.0])
    assert bench.parity_vs_n1(a, 1000, 0, tr)[0] is None                      # no fixture yet
    bench.write_fixture(a, 1000, 0, tr)
    assert bench.parity_vs_n1(a, 1000, 0, tr) == (0.0, "first 3 iterations; within 1e-10 over the first 3")
    rel, _ = bench.parity_vs_n1(a, 1000, 0, tr * (1 + 1e-12))
    assert 0 < rel < 2e-12
    assert bench.parity_vs_n1(a, 1000, 30, tr)[0] is None                     # another configuration
    rel, note = bench.parity_vs_n1(a, 1000, 0, tr * np.array([1.0, 1 + 1e-12, 1 + 1e-9]))
    assert rel > bench.PARITY_TOL and note.endswith("over the first 2")
    a.no_parity_assert = False
    bench.parity_gate(a, 1e-11, "x")
    bench.parity_gate(a, None, "x")
    import pytest
    with pytest.raises(AssertionError):
        bench.parity_gate(a, rel, "x")
    a.no_parity_assert = True
    bench.parity_gate(a, rel, "x")


def test_dump_outputs_sample_and_files(bench, tmp_path):
    import numpy as np
    assert np.array_equal(bench.sample_index(10, 16), np.arange(10))
    i = bench.sample_index(200_000_000, 1000)
    assert np.array_equal(i, bench.sample_index(200_000_000, 1000))                # seeded: the same entries every run
    assert len(i) == 1000 and np.all(np.diff(i) > 0) and i[-1] < 200_000_000
    bench.write_outputs(str(tmp_path / "o"), {"x": np.arange(3), "y": np.ones(2, np.float32)}, 0, 1)
    assert np.load(tmp_path / "o" / "x.npy").dtype == np.float64 and np.load(tmp_path / "o" / "y.npy").dtype == np.float32
    bench.write_outputs(str(tmp_path / "r"), {"x": np.zeros(2)}, 1, 2)
    assert os.listdir(tmp_path / "r") == ["x_rank1.npy"]
    with pytest.raises(AssertionError):
        bench.write_outputs(str(tmp_path / "big"), {"x": np.zeros(bench.DUMP_LIMIT // 8 + 1)}, 0, 1)
    assert not os.path.exists(tmp_path / "big")


@pytest.mark.gpu
def test_dump_outputs_of_two_runs_are_identical(tmp_path):
    import numpy as np

    def run(d):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "4", "--warmup", "3", "--n", "200000",
                            "--no-e2e", "--no-cpu-baseline", "--dump-outputs", str(d)],
                           capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stderr[-2000:]
        return json.loads(p.stdout.strip().splitlines()[-1])

    a, _ = run(tmp_path / "a"), run(tmp_path / "b")
    assert a["steps"] == 4 and a["config"]["repetitions"] == 1 and a["config"]["fdf_evals_in_timed_region"] >= 4
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b"))
    assert {"minimizer.npy", "gradient.npy", "objective.npy", "secondary_minimizer.npy"} <= set(names)
    for f in names:
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)), f
    if a["config"]["restarts_in_timed_region"] == 0:
        assert len(np.load(tmp_path / "a" / "trace_objective.npy")) == 3 + 4
    assert len(np.load(tmp_path / "a" / "minimizer.npy")) == 200_000
