"""Timing of the column sweep with and without pruning (option "col_prune", SdpTables.col_bound)
on config #5 (storage + AR(1), 2000 x 500 states, <= 256 controls, W = 9, layout CF).

The bench's trajectory: J from default_rng(0).standard_normal, 5 warm-up sweeps, 20 timed
device-resident sweeps (Engine.sweep), CUDA events around each streaming-kernel launch and
around the whole loop.  col_prune 0 and 1 alternate in the same process, --reps times each,
every repetition from the same J and with no seeds (part_idx = -1).  Reported per setting:
kernel and step times (median and range over the repetitions), the J and argmin of the last
sweep compared bit for bit between the settings, and - from a separate, untimed pass with the
opt-in counter "col_prune_stats" - the share of warp steps skipped in each sweep.  One JSON
document on stdout (and in --out), with the device name and power limit.

    python scripts/prune_timing.py [--reps 5] [--out profiles/r3_prune_timing.json]
"""
import argparse
import contextlib
import ctypes
import io
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def quiet(fn):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn()


def device_info(torch):
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        info["power_limit_and_max_sm_clock"] = q[0] if q else None
    except (OSError, subprocess.SubprocessError):
        info["power_limit_and_max_sm_clock"] = None
    return info


def run(torch, eng, T, J0, n, warmup, steps, prune, stats=False):
    """the bench's trajectory with col_prune = prune; returns (kernel ms [steps], loop ms, last J,
    last argmin, per-sweep (steps, skipped) when `stats`)"""
    from stodynprog_b200 import _cabi
    lib = eng.lib
    lib.sdp_set_option(b"col_prune", prune)
    lib.sdp_set_option(b"col_prune_stats", 1 if stats else 0)
    T.part_idx.fill_(-1)
    J_prev, J_new = eng.J_pair(n)
    eng.begin_call(n)
    eng.upload_J(J0, J_prev)
    counts = []

    def count():
        a, b = ctypes.c_int64(), ctypes.c_int64()
        _cabi.check(lib.sdp_col_prune_counts(ctypes.byref(a), ctypes.byref(b)), "sdp_col_prune_counts")
        return a.value, b.value

    if stats:
        count()
    for _ in range(warmup):
        eng.sweep(T, J_prev, J_new, defer_wait=True)
        J_prev, J_new = J_new, J_prev
        if stats:
            counts.append(count())
    eng.flush_exchange()
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    for k in range(steps):
        eng.sweep(T, J_prev, J_new, events=kev[k], defer_wait=True, want_argmin=(k == steps - 1))
        J_prev, J_new = J_new, J_prev
        if stats:
            counts.append(count())
    eng.flush_exchange()
    end.record()
    torch.cuda.synchronize()
    kernel = np.array([a.elapsed_time(b) for a, b in kev])
    lib.sdp_set_option(b"col_prune", 1)
    lib.sdp_set_option(b"col_prune_stats", 0)
    return kernel, start.elapsed_time(end), J_prev.cpu().numpy().copy(), T.argmin.cpu().numpy().copy(), counts


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("prune_timing.py measures on the GPU; no CUDA device found")
    import stodynprog_b200 as pkg
    import workloads as wl
    from stodynprog_b200 import _cabi

    class _Api(object):
        SysDescription = pkg.SysDescription

        def DPSolver(self, sys_, **kw):
            return pkg.DPSolver(sys_, **kw)

    sv = quiet(lambda: wl.storage_ar1_large(_Api()).solver)
    T = quiet(sv.sweep_tables)
    assert T.layout_name == "column_factored", T.layout_name
    eng = sv.engine
    n = int(np.prod(sv._state_grid_shape))
    J0 = np.random.default_rng(0).standard_normal(sv._state_grid_shape)

    res = {0: [], 1: []}
    last = {}
    kernel_name = {}
    for rep in range(args.reps):
        for prune in (0, 1) if rep % 2 == 0 else (1, 0):
            k, loop, J, A, _ = run(torch, eng, T, J0, n, args.warmup, args.steps, prune)
            kernel_name[prune] = _cabi.last_kernel()
            res[prune].append((float(np.mean(k)), loop / args.steps))
            if prune in last:
                assert np.array_equal(last[prune][0].view(np.int64), J.view(np.int64))
            last[prune] = (J, A)
    _, _, J, A, counts = run(torch, eng, T, J0, n, args.warmup, args.steps, 1, stats=True)
    same_J = bool(np.array_equal(last[0][0].view(np.int64), last[1][0].view(np.int64)))
    same_A = bool(np.array_equal(last[0][1], last[1][1]))
    counted_same = bool(np.array_equal(J.view(np.int64), last[1][0].view(np.int64)) and np.array_equal(A, last[1][1]))

    def summary(rows):
        k = np.array([r[0] for r in rows])
        s = np.array([r[1] for r in rows])
        return {"kernel_ms_median": round(float(np.median(k)), 4),
                "kernel_ms_range": [round(float(k.min()), 4), round(float(k.max()), 4)],
                "step_ms_median": round(float(np.median(s)), 4),
                "step_ms_range": [round(float(s.min()), 4), round(float(s.max()), 4)],
                "backups_per_s_median": float(T.n_backups_total / (np.median(s) * 1e-3))}

    share = [round(b / a, 4) if a else None for a, b in counts]
    out = dict(device_info(torch))
    out.update({
        "workload": "config #5: storage + AR(1), 2000 x 500 states, <= 256 controls, W = 9, layout CF, 1 GPU",
        "backups_per_sweep": int(T.n_backups_total),
        "trajectory": "J = default_rng(0).standard_normal; %d warm-up + %d timed device-resident sweeps, "
                      "part_idx = -1 at the start; settings alternated, %d repetitions each"
                      % (args.warmup, args.steps, args.reps),
        "kernel": {"col_prune=0": kernel_name[0], "col_prune=1": kernel_name[1]},
        "col_prune=0": summary(res[0]),
        "col_prune=1": summary(res[1]),
        "speedup_step_median": round(float(np.median([r[1] for r in res[0]]) / np.median([r[1] for r in res[1]])), 3),
        "last_sweep_bit_identical": {"J": same_J, "argmin": same_A, "with_counter_on": counted_same},
        "skipped_share_per_sweep": share,
        "skipped_share_timed_sweeps_mean": round(float(np.mean([x for x in share[args.warmup:] if x is not None])), 4),
        "skipped_share_note": "warp steps (col_ub controls of one item for 32 lanes) whose evaluation was "
                              "skipped, over all warp steps; counted in a separate untimed pass",
    })
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    if not (same_J and same_A and counted_same):
        sys.exit("pruning changed the results")


if __name__ == "__main__":
    main()
