"""Timing of the risk-averse sweeps (MeanCVaR, sdp_sweep_risk_partials) against the expectation.

Config #5 (storage + AR(1), 2000 x 500, <= 256 controls, W = 9): ms per sweep (streaming pass +
combine, one rank, J on the device) of
  - risk=None and MeanCVaR(0.9, 0.5) on the tables the solver picks (layout CF, which the risk
    sweep shares: k_sweep_risk_column after the column-table pre-pass),
  - risk=None and MeanCVaR(0.9, 0.5) on dense layout-A tables (k_sweep_risk<2,9>),
alternated round by round on the same J after a warm-up, from CUDA events; the set-up time and
device bytes of both table sets; value_iteration end to end with risk (host J in, host J and
policy out; tables cached).  Config #4 (SEAREV 31 x 61 x 61, W = 9): its default tables are
layout AF, which the risk sweep does not take: the risk sweep builds dense layout-A tables; the
expectation on the AF and on those tables, the risk on those.  The fp64 operations per (x,u) are
counted from the arithmetic contract (include/sdp_b200.h).  One JSON document on stdout (and in --out).

    python scripts/risk_timing.py [--sweeps 20] [--rounds 5] [--out profiles/r7_risk_timing.json]
"""
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

from first_passage_timing import quiet  # noqa: E402


def ops_per_xu(d, W, WM):
    """fp64 operations per (x,u) from the contract: node values (nested lerp 3 per level pair,
    g + v), the ordered expectation (W products, W sums); for the risk backup also the sort
    network (WM rounds of floor(WM/2) or floor((WM-1)/2) compare-exchanges, one or two fp64
    compares each: counted as 2), the walk (at most 4 per node: compare, subtract, product,
    sum; plus the cum update) and the combination (3)"""
    values = W * (3 * (2 ** d - 1) + 1)
    expect = values + 2 * W
    pairs = sum(len(range(r & 1, WM - 1, 2)) for r in range(WM))
    risk = expect + 2 * pairs + 5 * W + 1 + 3
    return expect, risk


def time_sweeps(torch, eng, cases, J0, sweeps, rounds):
    Jp, Jn = eng.J_pair(J0.numel())
    for T, r in cases.values():                               # warm-up
        for _ in range(3):
            Jp.copy_(J0)
            eng.sweep(T, Jp, Jn, risk=r)
    torch.cuda.synchronize()
    times = {k: [] for k in cases}
    for _ in range(rounds):
        for key, (T, r) in cases.items():
            Jp.copy_(J0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(sweeps):
                eng.sweep(T, Jp, Jn, risk=r)                  # the same J every sweep
            e1.record()
            e1.synchronize()
            times[key].append(e0.elapsed_time(e1) / sweeps)
    return times


def timed(torch, fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    T = quiet(fn)
    torch.cuda.synchronize()
    return T, time.perf_counter() - t0


def dense_a(solver):
    """dense layout-A tables of the solver's problem (what a risk sweep uses where CF does not apply)"""
    saved = solver.table_layout, solver.table_compress, solver.column_hoist
    solver.table_layout, solver.table_compress, solver.column_hoist = "control_minor", "off", "off"
    try:
        return solver.engine.build_sweep_tables(solver, None)
    finally:
        solver.table_layout, solver.table_compress, solver.column_hoist = saved


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sweeps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("risk_timing.py measures on a GPU; none is visible")
    import stodynprog_b200 as sdp
    import workloads as wl
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    res = {"device": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "",
           "risk": "MeanCVaR(alpha=0.9, weight=0.5)", "sweeps_per_round": args.sweeps, "rounds": args.rounds,
           "configs": []}
    R = sdp.MeanCVaR(0.9, 0.5)
    cR = R.c_struct()
    for name, make in (("#5 storage_ar1_large 2000x500", lambda: wl.storage_ar1_large(sdp)),
                       ("#4 searev 31x61x61", lambda: wl.searev(sdp))):
        prob = make()
        sv = prob.solver
        eng = sv.engine
        shape = sv._state_grid_shape
        J0 = eng.to_device(np.random.default_rng(0).standard_normal(shape).reshape(-1))
        T_e, t_e = timed(torch, lambda: sv.sweep_tables(None))
        T_r, t_r = timed(torch, lambda: sv.sweep_tables(None, risk=True))
        T_a, t_a = (T_r, t_r) if not T_r.column else timed(torch, lambda: dense_a(sv))
        cases = {"expectation_" + T_e.layout_name: (T_e, None)}
        if T_r is T_e:
            cases["risk_" + T_e.layout_name] = (T_e, cR)
        cases["expectation_" + T_a.layout_name] = (T_a, None)
        cases["risk_" + T_a.layout_name] = (T_a, cR)
        times = time_sweeps(torch, eng, cases, J0, args.sweeps, args.rounds)
        d, W = T_a.d, T_a.W
        n_xu = int(T_a.n_backups_total) // W if hasattr(T_a, "n_backups_total") else None
        e_ops, r_ops = ops_per_xu(d, W, 9 if W <= 9 else 16)
        out = {"config": name, "states": int(np.prod(shape)), "W": W, "d": d,
               "xu_pairs": n_xu, "tables": {}, "sweep_ms": {},
               "fp64_ops_per_xu": {"expectation": e_ops, "risk": r_ops}}
        out["risk_tables_shared_with_expectation"] = T_r is T_e
        for key, T, t in (("default", T_e, t_e), ("risk", T_r, t_r if T_r is not T_e else 0.0),
                          ("dense_A", T_a, t_a)):
            out["tables"][key] = {"layout": T.layout_name, "device_bytes": int(T.device_bytes), "setup_s": t}
        for key, ts in times.items():
            out["sweep_ms"][key] = {"median": float(np.median(ts)), "rounds": [float(x) for x in ts]}
        ms = {k: v["median"] for k, v in out["sweep_ms"].items()}
        for lay in {T_e.layout_name, T_a.layout_name}:
            if "risk_" + lay in ms:
                out["risk_over_expectation_" + lay] = ms["risk_" + lay] / ms["expectation_" + lay]
                if n_xu:
                    out["risk_fp64_rate_GFLOPs_" + lay] = n_xu * r_ops / (ms["risk_" + lay] * 1e-3) / 1e9
        if "risk_column_factored" in ms:
            # keep the CF risk kernel only if it beats layout-A risk on the same problem
            out["cf_risk_over_a_risk"] = ms["risk_column_factored"] / ms["risk_control_minor"]
        if name.startswith("#5"):
            Jh = np.random.default_rng(1).standard_normal(shape)
            quiet(lambda: sv.value_iteration(Jh, report_time=False, risk=R))        # warm
            e2e = []
            for _ in range(3):
                t0 = time.perf_counter()
                quiet(lambda: sv.value_iteration(Jh, report_time=False, risk=R))
                e2e.append(time.perf_counter() - t0)
            out["value_iteration_risk_e2e_s"] = {"median": float(np.median(e2e)), "runs": e2e}
        res["configs"].append(out)
        sv.clear_tables()
        del T_e, T_r, T_a, cases
        torch.cuda.empty_cache()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
