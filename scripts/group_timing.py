"""Timing of the column sweep with group skipping (sdp_column_groups_build, option "col_groups") on
config #5 (storage + AR(1), 2000 x 500 states, <= 256 controls, W = 9, layout CF).

The bench's trajectory, as scripts/prune_timing.py: J from default_rng(0).standard_normal, 5 warm-up
sweeps, 20 timed device-resident sweeps, CUDA events around each streaming-kernel launch and around
the whole loop, every repetition from the same J and with no seeds.  Settings, alternated --reps
times: no pruning, pruning without groups, pruning with groups of each K in --ks (the summaries are
rebuilt for each K).  Reported per setting: kernel and step times (median and range), the J and
argmin of the last sweep compared bit for bit, and - from a separate, untimed pass with the counter
"col_prune_stats" - per sweep the share of groups passed over, the share of warp steps skipped, and
the HBM bytes the sweep reads (summaries of the groups met, the (x,u) stream of the surviving
groups, tables and bounds), set against the device-to-device copy bandwidth measured in the same
run.  One JSON document on stdout (and in --out), with the device name and power limit.

    python scripts/group_timing.py [--reps 3] [--ks 8,16] [--out profiles/r7_group_timing.json]
"""
import argparse
import ctypes
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from prune_timing import device_info, quiet  # noqa: E402


def run(torch, eng, T, J0, n, warmup, steps, prune, groups, stats=False):
    """the bench's trajectory; returns (kernel ms [steps], loop ms, last J, last argmin, per-sweep
    (steps, skipped, groups, groups skipped) when `stats`)"""
    from stodynprog_b200 import _cabi
    lib = eng.lib
    lib.sdp_set_option(b"col_prune", prune)
    lib.sdp_set_option(b"col_groups", groups)
    lib.sdp_set_option(b"col_prune_stats", 1 if stats else 0)
    T.part_idx.fill_(-1)
    J_prev, J_new = eng.J_pair(n)
    eng.begin_call(n)
    eng.upload_J(J0, J_prev)
    counts = []

    def count():
        c = [ctypes.c_int64() for _ in range(4)]
        _cabi.check(lib.sdp_col_prune_counts(ctypes.byref(c[0]), ctypes.byref(c[1])), "sdp_col_prune_counts")
        _cabi.check(lib.sdp_col_group_counts(ctypes.byref(c[2]), ctypes.byref(c[3])), "sdp_col_group_counts")
        return [x.value for x in c]

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
    lib.sdp_set_option(b"col_groups", 1)
    lib.sdp_set_option(b"col_prune_stats", 0)
    return kernel, start.elapsed_time(end), J_prev.cpu().numpy().copy(), T.argmin.cpu().numpy().copy(), counts


def copy_bandwidth(torch, nbytes=2 << 30, reps=10):
    """device-to-device copy of nbytes: bytes read + written per second"""
    a = torch.empty(nbytes // 8, dtype=torch.float64, device="cuda")
    b = torch.empty_like(a)
    for _ in range(2):
        b.copy_(a)
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    s.record()
    for _ in range(reps):
        b.copy_(a)
    e.record()
    torch.cuda.synchronize()
    return 2.0 * nbytes * reps / (s.elapsed_time(e) * 1e-3)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--ks", default="8,16")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("group_timing.py measures on the GPU; no CUDA device found")
    import stodynprog_b200 as pkg
    import workloads as wl
    from stodynprog_b200 import _cabi, tablebuild

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
    ks = [int(k) for k in args.ks.split(",")]
    rows = sv._state_grid_shape[0]
    table_bytes = T.n_cols * (8 * _cabi.column_pitch(rows, T.W) + 16 * rows)
    pairs = int(T.item_u_count_host.sum()) * 32          # (x,u) pairs of the stream, padding included

    settings = [("col_prune=0", 0, 0, None), ("col_prune=1,col_groups=0", 1, 0, None)] + \
        [("col_prune=1,col_groups=1,K=%d" % k, 1, 1, k) for k in ks]
    res, last, kname, info = {}, {}, {}, {}
    for rep in range(args.reps):
        order = settings if rep % 2 == 0 else settings[::-1]
        for name, prune, groups, k in order:
            if k is not None:
                tablebuild.build_column_groups(eng, T, k)
                Kc, Lc = ctypes.c_int32(), ctypes.c_int32()
                eng.lib.sdp_column_groups_info(T.col_groups_id, ctypes.byref(Kc), ctypes.byref(Lc))
                info[name] = {"K": Kc.value, "L": Lc.value, "summary_bytes": int(T.col_groups.numel())}
            kt, loop, J, A, _ = run(torch, eng, T, J0, n, args.warmup, args.steps, prune, groups)
            kname[name] = _cabi.last_kernel()
            res.setdefault(name, []).append((float(np.mean(kt)), loop / args.steps))
            last[name] = (J, A)
    bw = copy_bandwidth(torch)
    ref_J, ref_A = last["col_prune=0"]
    out = dict(device_info(torch))
    out.update({
        "workload": "config #5: storage + AR(1), 2000 x 500 states, <= 256 controls, W = 9, layout CF, 1 GPU",
        "backups_per_sweep": int(T.n_backups_total),
        "trajectory": "J = default_rng(0).standard_normal; %d warm-up + %d timed device-resident sweeps, "
                      "part_idx = -1 at the start; settings alternated, %d repetitions each"
                      % (args.warmup, args.steps, args.reps),
        "copy_bandwidth_TBps": round(bw / 1e12, 3),
        "settings": {},
    })
    ok = True
    for name, prune, groups, k in settings:
        rows_ = res[name]
        kt = np.array([r[0] for r in rows_])
        st = np.array([r[1] for r in rows_])
        J, A = last[name]
        same = bool(np.array_equal(J.view(np.int64), ref_J.view(np.int64)) and np.array_equal(A, ref_A))
        ok &= same
        entry = {"kernel": kname[name],
                 "kernel_ms_median": round(float(np.median(kt)), 4),
                 "kernel_ms_range": [round(float(kt.min()), 4), round(float(kt.max()), 4)],
                 "step_ms_median": round(float(np.median(st)), 4),
                 "step_ms_range": [round(float(st.min()), 4), round(float(st.max()), 4)],
                 "last_sweep_bit_identical_to_col_prune_0": same}
        if prune:
            if k is not None:
                tablebuild.build_column_groups(eng, T, k)
                entry.update(info[name])
            _, _, J2, A2, counts = run(torch, eng, T, J0, n, args.warmup, args.steps, prune, groups, stats=True)
            ok &= bool(np.array_equal(J2.view(np.int64), ref_J.view(np.int64)) and np.array_equal(A2, ref_A))
            entry["skipped_warp_step_share_per_sweep"] = [round(c[1] / c[0], 4) if c[0] else None for c in counts]
            if k is not None:
                entry["skipped_group_share_per_sweep"] = [round(c[3] / c[2], 4) if c[2] else None for c in counts]
                # summaries of the groups met (512 B each) + 20 B per pair of the surviving groups
                read = [c[2] * 512 + (c[2] - c[3]) * k * 32 * 20 + table_bytes for c in counts]
            else:
                read = [pairs * 20 + table_bytes for _ in counts]
            entry["hbm_bytes_read_per_sweep_GB"] = [round(r / 1e9, 3) for r in read]
            mean_read = float(np.mean(read[args.warmup:]))
            entry["hbm_bytes_read_timed_mean_GB"] = round(mean_read / 1e9, 3)
            entry["hbm_TBps_at_kernel_median"] = round(mean_read / (np.median(kt) * 1e-3) / 1e12, 3)
            entry["hbm_frac_of_copy_bandwidth"] = round(mean_read / (np.median(kt) * 1e-3) / bw, 3)
        out["settings"][name] = entry
    base = np.median([r[1] for r in res["col_prune=1,col_groups=0"]])
    out["speedup_step_median_vs_col_groups_0"] = {
        name: round(float(base / np.median([r[1] for r in res[name]])), 3) for name, _, g, _ in settings if g}
    out["hbm_bytes_note"] = ("bytes the streaming kernel reads per sweep, from the counters: 512 B of summaries per "
                             "group met, 20 B (cell, g, lambda0) per (x,u) pair of a surviving group, the column "
                             "tables and bounds; the pre-pass is not counted")
    tablebuild.build_column_groups(eng, T)
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    if not ok:
        sys.exit("group skipping changed the results")


if __name__ == "__main__":
    main()
