"""Timing of the forward operator (DPSolver.propagate_distribution / stationary_distribution)
on configs #5 (storage + AR(1), 2000 x 500, W = 9; policy of one value_iteration from zeros) and
#4 (SEAREV 31 x 61 x 61, W = 9; the reference's policy-iteration policy, tests/golden).

Per config: CSR build time (sdp_forward_build, after one warm-up build), time per step from CUDA
events over >= 1000 steps after a warm-up, the bytes a step must move and the achieved fraction
of the device-to-device copy bandwidth measured in the same run, and one scipy step on the host
over the same matrix.  One JSON document on stdout (and in --out).

    python scripts/forward_timing.py [--steps 2000] [--out results/forward_timing.json]
"""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def quiet(fn):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn()


def copy_bandwidth(torch, nbytes=2 << 30, reps=20):
    """device-to-device copy rate, (read + write) bytes per second"""
    a = torch.empty(nbytes // 8, dtype=torch.float64, device="cuda")
    b = torch.empty_like(a)
    a.fill_(1.0)
    for _ in range(3):
        b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        b.copy_(a)
    e1.record()
    e1.synchronize()
    return 2.0 * nbytes * reps / (e0.elapsed_time(e1) * 1e-3)


def measure(torch, name, solver, pol, steps, copy_bw):
    import scipy.sparse as sp
    eng = solver.engine
    P = quiet(lambda: eng.build_policy_tables(solver, pol, deterministic=True))
    F = eng.build_forward(P)                                  # warm-up build
    del F
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    F = eng.build_forward(P)                                  # ends with a read-back: synchronised
    t_build = time.perf_counter() - t0
    n, nnz = F.n, F.nnz
    mu_a = torch.full((n,), 1.0 / n, dtype=torch.float64, device="cuda")
    mu_b = torch.empty_like(mu_a)
    cost = torch.empty(steps, dtype=torch.float64, device="cuda")
    eng.forward_steps(F, mu_a, mu_b, 100, cost)               # warm-up
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    eng.forward_steps(F, mu_a, mu_b, steps, cost)
    e1.record()
    e1.synchronize()
    t_step = e0.elapsed_time(e1) * 1e-3 / steps
    # what one step must move: src + coef of every entry, row_ptr + piece_first, mu_in (read
    # twice: gathers, at least once, and the cost / residual terms), g_bar, mu_out
    bytes_step = 12 * nnz + 16 * (n + 1) + 8 * n * 4
    # host comparison: one scipy CSR product over the same matrix (rows = destinations)
    rp = F.bufs["row_ptr"].cpu().numpy()
    src = F.bufs["src"].cpu().numpy()
    coef = F.bufs["coef"].cpu().numpy()
    A = sp.csr_matrix((coef, src, rp), shape=(n, n))
    mu = np.full(n, 1.0 / n)
    A @ mu
    t0 = time.perf_counter()
    A @ mu
    t_scipy = time.perf_counter() - t0
    return {"config": name, "states": n, "W": P.W, "d": P.grid.d, "nnz": nnz,
            "long_row_pieces": F.n_pieces,
            "csr_build_s": t_build, "steps_timed": steps, "step_us": t_step * 1e6,
            "bytes_per_step": bytes_step, "achieved_TBps": bytes_step / t_step / 1e12,
            "fraction_of_copy_bw": bytes_step / t_step / copy_bw,
            "csr_bytes": 12 * nnz + 8 * (n + 1),
            "scipy_host_step_ms": t_scipy * 1e3, "speedup_vs_scipy_step": t_scipy / t_step}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("forward_timing.py measures on a GPU; none is visible")
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
    res["configs"].append(measure(torch, "#5 storage_ar1_large 2000x500", prob.solver, pol, args.steps, copy_bw))
    prob = wl.searev(sdp)
    res["configs"].append(measure(torch, "#4 searev 31x61x61", prob.solver, golden("searev_full.npz")["pi_pol"],
                                  args.steps, copy_bw))
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
