"""Timing of the path sampler (DPSolver.sample_paths: sdp_chain_pack + sdp_chain_sample) on
configs #5 (storage + AR(1), 2000 x 500, W = 9; policy of one value_iteration from zeros) and #4
(SEAREV 31 x 61 x 61, W = 9; the reference's policy-iteration policy, tests/golden).

Per config: 10^6 paths x 1000 steps from the uniform distribution, with a target set (axis 0 at
its lowest level) and no recorded steps, timed with CUDA events around the sampling launch after
a warm-up launch, three times.  Reported: transitions per second, the bytes of the 32-byte sectors
a transition reads from its packed record (a random access: 32 for d <= 2, 64 for d = 3, 4) times
that rate over the device-to-device copy bandwidth measured in the same run, and the numpy twin's
transitions per second on the host for 10^4 paths.  The card's name and power limit are read in the
same run.  One JSON document on stdout (and in --out).

    python scripts/sample_paths_timing.py [--paths 1000000] [--steps 1000] [--out results/x.json]
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


def measure(torch, name, solver, pol, M, steps, copy_bw):
    import chain_twin
    from stodynprog_b200 import _cabi
    eng = solver.engine
    dims = solver._state_grid_shape
    n = int(np.prod(dims))
    P = quiet(lambda: eng.build_policy_tables(solver, pol, deterministic=True))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    C = eng.chain_tables(P)
    torch.cuda.synchronize()
    t_pack = time.perf_counter() - t0
    d = P.grid.d
    target = np.zeros(dims, dtype=bool)
    target[0] = True
    mask = eng.to_device(solver._target_mask(target))
    start_cdf = eng.to_device(np.cumsum(np.ones(n)))
    state = torch.empty(M, dtype=torch.int32, device="cuda")
    total = torch.empty(M, dtype=torch.float64, device="cuda")
    hit = torch.empty(M, dtype=torch.int32, device="cuda")
    cnt = torch.zeros(2, dtype=torch.int64, device="cuda")
    eng.chain_sample(C, state, total, hit, 50, 0, 1, True, cnt, start_cdf=start_cdf, target=mask)   # warm-up
    times = []
    for rep in range(3):
        cnt.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        eng.chain_sample(C, state, total, hit, steps, 0, 1000 + rep, True, cnt, start_cdf=start_cdf, target=mask)
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1) * 1e-3)
    clamped = int(cnt[0].item())
    t = min(times)
    rate = M * steps / t
    rec_bytes = 8 * _cabi.chain_rec(d)
    sector_bytes = 32 if rec_bytes == 32 else 64      # a 48-byte record always spans two sectors
    # the twin on the host: 10^4 paths x 20 steps on the device's records
    orders = list(P.grid.order[:d])
    strides = [int(np.prod(orders[k + 1:])) for k in range(d)]
    rec = C.rec.cpu().numpy().reshape(-1, _cabi.chain_rec(d))
    m, k = 10000, 20
    st, tot, h = np.zeros(m, np.int32), np.zeros(m), np.zeros(m, np.int32)
    t0 = time.perf_counter()
    chain_twin.sample(strides, C.W, C.cdf.cpu().numpy(), rec, n, k, 0, 1, True, st, tot, h, [0, 0],
                      start_cdf=np.cumsum(np.ones(n)))
    t_twin = time.perf_counter() - t0
    return {"config": name, "states": n, "W": P.W, "d": d, "record_bytes": rec_bytes,
            "records_MB": n * P.W * rec_bytes / 1e6, "pack_s": t_pack, "paths": M, "steps": steps,
            "sample_s": times, "transitions_per_s": rate, "G_transitions_per_s": rate / 1e9,
            "sector_bytes_per_transition": sector_bytes,
            "sector_TBps": rate * sector_bytes / 1e12, "fraction_of_copy_bw": rate * sector_bytes / copy_bw,
            "clamped_share": clamped / (M * steps), "kernel": _cabi.last_kernel(),
            "twin_host_transitions_per_s": m * k / t_twin, "speedup_vs_twin": rate / (m * k / t_twin)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--paths", type=int, default=1000000)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("sample_paths_timing.py measures on a GPU; none is visible")
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
    res["configs"].append(measure(torch, "#5 storage_ar1_large 2000x500", prob.solver, pol, args.paths,
                                  args.steps, copy_bw))
    prob = wl.searev(sdp)
    res["configs"].append(measure(torch, "#4 searev 31x61x61", prob.solver, golden("searev_full.npz")["pi_pol"],
                                  args.paths, args.steps, copy_bw))
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
