"""Timing of the cost-moment recursion (DPSolver.cost_moments, sdp_cost_moments) on configs #5
(storage + AR(1), 2000 x 500, W = 9; policy of one value_iteration from zeros) and #4 (SEAREV
31 x 61 x 61, W = 9; the reference's policy-iteration policy, tests/golden).

Per config, on the same policy tables: the time per step of k_cost_moments (clamped weights and
unclamped, no target), of k_first_passage (clamped, target axis-0 index 0) and of an eval_policy
step (k_policy_eval), from CUDA events over rounds of --steps steps each, the four kernels
alternated round by round after a warm-up; the bytes a step must stream (the tables once) and the
achieved fraction of the device-to-device copy rate measured in the same run.  One JSON document
on stdout (and in --out).

    python scripts/cost_moments_timing.py [--steps 500] [--rounds 4] [--out results/cm.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from first_passage_timing import quiet  # noqa: E402  (scripts/ is on sys.path when run as a script)
from forward_timing import copy_bandwidth  # noqa: E402


def measure(torch, name, solver, pol, steps, rounds, copy_bw):
    eng = solver.engine
    dims = solver._state_grid_shape
    target = np.zeros(dims, dtype=bool)
    target[0] = True
    P = quiet(lambda: eng.build_policy_tables(solver, np.asarray(pol, dtype=float), deterministic=True))
    n, W, d = P.n_states, P.W, P.grid.d
    mask = eng.to_device(solver._target_mask(target))
    Va, Vb = torch.zeros(4 * n, dtype=torch.float64, device="cuda"), torch.empty(4 * n, dtype=torch.float64,
                                                                                 device="cuda")
    Ja, Jb = torch.zeros(n, dtype=torch.float64, device="cuda"), torch.empty(n, dtype=torch.float64, device="cuda")
    hist = torch.zeros(1, dtype=torch.float64, device="cuda")
    runs = {"cost_moments_clamp": lambda k: eng.cost_moments(P, None, True, Va, Vb, k),
            "cost_moments_noclamp": lambda k: eng.cost_moments(P, None, False, Va, Vb, k),
            "first_passage_clamp": lambda k: eng.first_passage(P, mask, True, Va, Vb, k),
            "eval_policy": lambda k: eng.policy_eval(P, Ja, Jb, k, False, 0, hist)}
    for fn in runs.values():                                   # warm-up
        fn(100)
    torch.cuda.synchronize()
    times = {k: [] for k in runs}
    for _ in range(rounds):
        for key, fn in runs.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn(steps)
            e1.record()
            e1.synchronize()
            times[key].append(e0.elapsed_time(e1) * 1e-3 / steps)
    # what a step must stream: the table planes (cell 4 B, lam 8d B, g 8 B per (x, w) entry or per
    # state), read once; then the values read (at least once) and written.  The second pass of
    # k_cost_moments reads the tables and gathers the corners again: not counted.
    tables = n * W * (4 + 8 * d) + 8 * n * (W if P.g_per_w else 1)
    rec_bytes = tables + 2 * 32 * n
    fp_bytes = rec_bytes + 4 * ((n + 31) // 32)
    ev_bytes = tables + 2 * 8 * n
    out = {"config": name, "states": n, "W": W, "d": d, "g_per_w": int(P.g_per_w), "steps_per_round": steps,
           "rounds": rounds, "cost_moments_target": "none", "first_passage_target": "axis-0 index 0",
           "table_bytes": tables}
    for key, ts in times.items():
        t = float(np.median(ts))
        b = ev_bytes if key == "eval_policy" else (fp_bytes if key.startswith("first") else rec_bytes)
        out[key] = {"step_us": t * 1e6, "step_us_rounds": [x * 1e6 for x in ts], "bytes_per_step": b,
                    "achieved_TBps": b / t / 1e12, "fraction_of_copy_bw": b / t / copy_bw}
    fp = out["first_passage_clamp"]["step_us"]
    ev = out["eval_policy"]["step_us"]
    for c in ("clamp", "noclamp"):
        out["ratio_%s_to_first_passage" % c] = out["cost_moments_" + c]["step_us"] / fp
        out["ratio_%s_to_eval_policy" % c] = out["cost_moments_" + c]["step_us"] / ev
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("cost_moments_timing.py measures on a GPU; none is visible")
    import stodynprog_b200 as sdp
    import workloads as wl
    from conftest import golden
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    copy_bw = copy_bandwidth(torch)
    res = {"device": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "",
           "copy_bw_TBps": copy_bw / 1e12, "configs": []}
    prob = wl.storage_ar1_large(sdp)
    _, pol = quiet(lambda: prob.solver.value_iteration(prob.J0, report_time=False))
    res["configs"].append(measure(torch, "#5 storage_ar1_large 2000x500", prob.solver, pol, args.steps,
                                  args.rounds, copy_bw))
    prob = wl.searev(sdp)
    res["configs"].append(measure(torch, "#4 searev 31x61x61", prob.solver, golden("searev_full.npz")["pi_pol"],
                                  args.steps, args.rounds, copy_bw))
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
