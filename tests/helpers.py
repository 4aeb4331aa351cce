"""Shared test helpers: config builders that create the SAME configuration for the oracle
(`oracle.make_config`) and for the host mirror (`cgoptim_b200` config objects)."""
from __future__ import annotations

import numpy as np

import cgoptim_b200 as cg
from oracle import oracle as O

FLAVOURS = ["HagerZhang", "YuanWangSheng", "SallehAlhawarat", "LiuStorrey", "LBFGS"]
LINESEARCHES = ["StrongWolfeBisection", "Wolfe", "YuanWeiLuWolfe", "Backtracking"]


def make_pair(flavour="HagerZhang", linesearch="StrongWolfeBisection", eps=1e-5, max_iters=1000,
              mu=0.1, lbfgs_m=10, c1=None, c2=None, delta1=1e-6, growth=2.0, ls_max_iters=None,
              zoom_max_iters=100, max_step_size=1e12, feas_max_iters=50, discount=0.9,
              sum_mode="cgo", beta_form="fused", trace=True):
    """Returns (oracle OrcConfig, host CGConfig, host LineSearchConfig).  Defaults follow the
    reference's examples (examples/min.jl:16-35, examples/constrained.jl:66-104)."""
    if linesearch == "StrongWolfeBisection":
        c1 = 1e-5 if c1 is None else c1
        c2 = 0.8 if c2 is None else c2
        ls_max_iters = 1000 if ls_max_iters is None else ls_max_iters
        ls = cg.setupStrongWolfeBisection(c1, c2, a_max_growth_factor=growth, max_iters=ls_max_iters,
                                          zoom_max_iters=zoom_max_iters)
    elif linesearch == "Wolfe":
        c1 = 1e-3 if c1 is None else c1
        c2 = 0.9 if c2 is None else c2
        ls_max_iters = 100 if ls_max_iters is None else ls_max_iters
        ls = cg.WolfeBisection(cg.Wolfe(c1, c2), ls_max_iters, max_step_size, feas_max_iters)
    elif linesearch == "YuanWeiLuWolfe":
        c1 = 1e-3 if c1 is None else c1
        c2 = 0.9 if c2 is None else c2
        ls_max_iters = 100 if ls_max_iters is None else ls_max_iters
        ls = cg.WolfeBisection(cg.YuanWeiLuWolfe(c1, c2, delta1), ls_max_iters, max_step_size, feas_max_iters)
    else:
        c1 = 1e-3 if c1 is None else c1
        c2 = 0.9 if c2 is None else c2
        ls_max_iters = 300 if ls_max_iters is None else ls_max_iters
        ls = cg.Backtracking(cg.Armijo(c1), discount, ls_max_iters, feas_max_iters)
    β = {"HagerZhang": cg.HagerZhang(), "YuanWangSheng": cg.YuanWangSheng(mu),
         "SallehAlhawarat": cg.SallehAlhawarat(), "LiuStorrey": cg.LiuStorrey(),
         "LBFGS": cg.LBFGS(lbfgs_m)}[flavour]
    cfg = cg.setupCGConfig(eps, β, cg.EnableTrace() if trace else cg.DisableTrace(), max_iters=max_iters)
    ocfg = O.make_config(flavour, linesearch, eps=eps, max_iters=max_iters, mu=mu, lbfgs_m=lbfgs_m,
                         c1=c1, c2=c2, delta1=delta1, growth=growth, ls_max_iters=ls_max_iters,
                         zoom_max_iters=zoom_max_iters, max_step_size=max_step_size,
                         feas_max_iters=feas_max_iters, discount=discount, sum_mode=sum_mode,
                         beta_form=beta_form)
    return ocfg, cfg, ls


def natural_lbfgs_rejection_case():
    """(oracle config, host config, line search, x0) of a run of the chained Rosenbrock (n = 2) with LBFGS(1) and
    Backtracking{Armijo}: Armijo alone does not keep s·y > 0, and from this start getβ rejects a pair while the
    one-pair history is full, after which the run goes on to max_iters"""
    ocfg, cfg, ls = make_pair("LBFGS", "Backtracking", eps=1e-10, max_iters=100, lbfgs_m=1)
    return ocfg, cfg, ls, np.array([2.1769160886969896, 2.6836698800822507])


def assert_same_run(ret, ora, exact=True, rtol=0.0, what=""):
    """Host-mirror Results vs OracleResult: statuses, counts, line-search decisions equal;
    f / ‖g‖ traces bit-identical (exact) or within rtol."""
    assert ret.status == ora.status, f"{what}: status {ret.status} != {ora.status}"
    assert ret.iters_ran == ora.iters_ran, f"{what}: iters {ret.iters_ran} != {ora.iters_ran}"
    t = ret.trace
    assert len(t.objective) == len(ora.trace_objective)
    assert np.array_equal(t.objective_evals, ora.trace_objective_evals), f"{what}: fdf evals differ"
    assert np.array_equal(t.step_size, ora.trace_step_size), f"{what}: step sizes differ"
    if exact:
        assert np.array_equal(t.objective, ora.trace_objective), f"{what}: objective trace differs"
        assert np.array_equal(t.grad_norm, ora.trace_grad_norm), f"{what}: grad-norm trace differs"
        assert (ret.objective == ora.objective) or (np.isnan(ret.objective) and np.isnan(ora.objective))
        assert np.array_equal(ret.minimizer, ora.minimizer, equal_nan=True), f"{what}: minimizer differs"
        assert np.array_equal(ret.gradient, ora.gradient, equal_nan=True), f"{what}: gradient differs"
    else:
        np.testing.assert_allclose(t.objective, ora.trace_objective, rtol=rtol)
        np.testing.assert_allclose(t.grad_norm, ora.trace_grad_norm, rtol=rtol)


def record_gate(name, **numbers):
    """Append the measured numbers of a tolerance gate to gpurun_out/north_star_gates.jsonl (brought back from the
    GPU box; the committed copy is profiles/r2_north_star_gates.jsonl, quoted in DESIGN.md §3)."""
    import json
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    os.makedirs(os.path.join(root, "gpurun_out"), exist_ok=True)
    rec = {"gate": name}
    rec.update({k: (float(v) if isinstance(v, (np.floating, float)) else (int(v) if isinstance(v, (np.integer, int)) else v))
                for k, v in numbers.items()})
    with open(os.path.join(root, "gpurun_out", "north_star_gates.jsonl"), "a") as f:
        f.write(json.dumps(rec) + "\n")
    print("GATE", json.dumps(rec))


def gate_numbers(ret, ora, ora2, m):
    """north_star's 1e-10 gate, measured: `window` = leading iterations on which two legitimate reference summation
    orders (ora: sequential, ora2: compensated) agree to 2.5e-11; max relative deviation of the device run from the
    sequential oracle inside the window, at iteration m, and overall over the first m iterations."""
    rel = lambda a, b: np.abs(np.asarray(a) / np.asarray(b) - 1.0)
    drift = np.maximum(rel(ora.trace_objective[:m], ora2.trace_objective[:m]), rel(ora.trace_grad_norm[:m], ora2.trace_grad_norm[:m]))
    bad = np.nonzero(drift > 2.5e-11)[0]
    w = int(bad[0]) if bad.size else m
    df, dg = rel(ret.trace.objective[:m], ora.trace_objective[:m]), rel(ret.trace.grad_norm[:m], ora.trace_grad_norm[:m])
    return w, dict(window=w, iterations_compared=m,
                   f_maxrel_in_window=df[:w].max(), g_maxrel_in_window=dg[:w].max(),
                   f_rel_at_last=df[m - 1], g_rel_at_last=dg[m - 1], f_maxrel_all=df.max(), g_maxrel_all=dg.max(),
                   reference_orders_f_rel_at_last=rel(ora.trace_objective[:m], ora2.trace_objective[:m])[m - 1],
                   reference_orders_g_rel_at_last=rel(ora.trace_grad_norm[:m], ora2.trace_grad_norm[:m])[m - 1],
                   decisions_identical=bool(np.array_equal(ret.trace.step_size[:m], ora.trace_step_size[:m])
                                            and np.array_equal(ret.trace.objective_evals[:m], ora.trace_objective_evals[:m])),
                   iters_device=int(ret.iters_ran), iters_oracle_seq=int(ora.iters_ran), iters_oracle_comp=int(ora2.iters_ran),
                   final_f_rel=abs(ret.objective - ora.objective) / max(abs(ora.objective), 1e-300))
