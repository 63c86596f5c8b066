"""Sharded-sweep parity check, to be launched with one process per GPU:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 \
        --master-addr 127.0.0.1 --master-port 29511 tests/multi_gpu_check.py

Every rank builds the tables of its slab of the storage-AR1 grid (config #3),
runs value_iteration / eval_policy / policy_iteration through the public API
(NCCL all-gather of J per sweep) and compares with the golden fixtures produced
by the unmodified reference.  Exit code 0 = parity on every rank."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def check_column_layout(sdp, wl, rank):
    """layout CF (one inner-interpolation table per grid column) over several ranks, the
    grid cut into whole rows and into whole columns, against the oracle port on the host"""
    from conftest import rel_err
    from oracle.ref_port import port_api
    world = dist.get_world_size()
    n_E, n_P = 32 * world + 8, 2 * world + 3
    kw = dict(n_E=n_E, n_P=n_P, n_w=9, steps=(0.5, 0.1))
    ora = wl.storage_ar1(port_api(), **kw).solver
    J0 = np.random.default_rng(5).standard_normal((n_E, n_P))
    want = []
    J = J0
    for k in range(2):
        J, pol = ora.value_iteration(J)
        want.append((J, pol))
    ok = True
    # (the cut by columns runs when asked for: SDP_CHECK_COLUMN_AXIS=1, as in profiles/r2_multi_gpu_check_n{2,8}.log;
    # tests/test_peer_exchange.py checks the same exchange with the ranks emulated on one GPU)
    axes = ("rows", "columns") if os.environ.get("SDP_CHECK_COLUMN_AXIS") else ("rows",)
    for axis in axes:
        sv = wl.storage_ar1(sdp, **kw).solver
        sv.table_layout = "state_minor"
        sv.column_hoist = "on"
        sv.slab_axis = axis
        J = J0
        for k in range(2):
            J, pol = sv.value_iteration(J, report_time=False)
            bad = int(np.any(pol != want[k][1], axis=-1).sum())
            err = rel_err(J, want[k][0])
            ok &= bad == 0 and err <= 1e-10
            if rank == 0:
                print("[column_factored, slabs of %s] sweep %d: policy mismatches %d, J rel err %.2e"
                      % (axis, k, bad, err))
        T = sv.last_tables
        ok &= T.column and (T.col_bounds is not None) == (axis == "columns")
        Js, pols, info = sv.solve_value_iteration(J_zero=J0, max_iter=2, tol=0.0)
        r_expected = np.max(np.abs(want[1][0] - want[0][0]))
        ok &= rel_err(Js, want[1][0]) <= 1e-10 and abs(info["residuals"][-1] - r_expected) <= 1e-9 * r_expected
        print("[column_factored, slabs of %s] rank %d: %d states, %s" % (
              axis, rank, T.n_states, "columns %s" % T.col_bounds if T.col_bounds else "bounds %s" % T.bounds),
              flush=True)
    return bool(ok)


def check_tiny_grid_and_late_peer(sdp, wl, rank):
    """the 10 states of the inventory problem (config #1) over all the ranks: some ranks hold one
    state, with eight ranks some hold NONE (an empty shard still has to publish its epoch), and
    one rank arrives a second late at every other sweep (its peers wait on their flags); against
    the golden fixture of the unmodified reference"""
    import time
    from conftest import golden, rel_err
    G = golden("inventory.npz")
    prob = wl.inventory(sdp)
    J, ok = prob.J0, True
    for k in range(6):
        if k % 2 == 1 and rank == dist.get_world_size() - 1:
            time.sleep(1.0)
        J, u = prob.solver.value_iteration(J, report_time=False)
        ok &= np.array_equal(u, G["pol"][k]) and rel_err(J, G["J"][k]) <= 1e-10
    T = prob.solver.last_tables
    sizes = [None] * dist.get_world_size()
    dist.all_gather_object(sizes, int(T.n_states))
    if rank == 0:
        print("[inventory, 10 states] states per rank %s, late peer tolerated: %s" % (sizes, "OK" if ok else "FAILED"),
              flush=True)
    return bool(ok)


def check_shared_results(sdp, wl, rank):
    """host results through the shared page-locked segment (hostshare.py): every array handed
    out keeps its values while it is alive - five sweeps whose results are all KEPT (the ring has
    three slots: the later calls must fall back to private copies, not overwrite), then a loop
    that drops them (slots recycled); rank 0's arrays are writable, the others' read-only"""
    from conftest import rel_err
    from oracle.ref_port import port_api
    from stodynprog_b200.hostshare import SlotArray
    kw = dict(steps=(0.05, 0.1))
    sv, so = wl.storage_ar1(sdp, **kw).solver, wl.storage_ar1(port_api(), **kw).solver
    J0 = np.random.default_rng(21).standard_normal(sv._state_grid_shape)
    kept, J, shared, fails = [], J0, 0, []

    def same_policy(J_in, pol_gpu, pol_port, what):
        """policies equal, or - counted and printed - different only where the port's own values
        of the two controls are tied to the last bits (the order of the expectation sum differs
        between np.inner and the kernel: north_star's 'exact ties counted and reported')"""
        bad = np.argwhere(np.any(pol_gpu != pol_port, axis=-1))
        if len(bad) == 0:
            return True
        Ji = so.interp_on_state(np.array(J_in))
        worst = 0.0
        for idx in bad:
            x_k = tuple(g[i] for g, i in zip(so.state_grid, idx))
            grids, dims = so.control_grids(x_k)
            _, _, flat, Jall = so.value_at_state(x_k, Ji, None, True)
            u_idx = tuple(int(np.argmin(np.abs(grids[c] - pol_gpu[tuple(idx)][c]))) for c in range(len(grids)))
            gap = abs(float(Jall[u_idx]) - float(Jall.reshape(-1)[flat])) / max(abs(float(Jall.reshape(-1)[flat])), 1e-300)
            worst = max(worst, gap)
        if rank == 0:
            print("[shared host results] %s: %d states with another control, tied within %.1e (relative)"
                  % (what, len(bad), worst), flush=True)
        return worst <= 1e-13

    def need(cond, what):
        if not cond:
            fails.append(what)
    for k in range(5):
        J, pol = sv.value_iteration(J, report_time=False)
        kept.append((J, pol))
        shared += isinstance(J, SlotArray)
    # (every sweep is checked against the port fed with the SAME input array, so that a
    # near-tie cannot be broken differently because of a last-bit difference in J)
    want = [so.value_iteration(np.array(J0 if k == 0 else kept[k - 1][0])) for k in range(5)]
    for k, (Jk, polk) in enumerate(kept):
        need(same_policy(J0 if k == 0 else kept[k - 1][0], polk, want[k][1], "kept sweep %d" % k), "kept policy %d" % k)
        need(rel_err(Jk, want[k][0]) <= 1e-10, "kept J %d (%.2e)" % (k, rel_err(Jk, want[k][0])))
    need(1 <= shared < 5, "%d of 5 kept results in shared slots" % shared)
    if isinstance(kept[0][0], SlotArray):
        need(kept[0][0].flags.writeable == (rank == 0), "writeable flag")
    del kept, pol, Jk, polk
    for k in range(5, 7):
        J_in = np.array(J)
        Jo, polo = so.value_iteration(J_in.copy())
        J, pol = sv.value_iteration(J, report_time=False)
        need(isinstance(J, SlotArray), "recycled slot %d" % k)
        need(same_policy(J_in, pol, polo, "sweep %d" % k) and rel_err(J, Jo) <= 1e-10, "values after recycling %d" % k)
    J_in = np.array(J) - J[sv._state_ref_ind]
    (Jd, Jr), pol = sv.value_iteration((J_in, 0.), rel_dp=True, report_time=False)
    (Jdo, Jro), polo = so.value_iteration((J_in.copy(), 0.), rel_dp=True)
    need(same_policy(J_in, pol, polo, "relative DP"), "relative DP policy")
    need(abs(Jr - Jro) <= 1e-10 * abs(Jro), "relative DP J_ref %r vs %r" % (Jr, Jro))
    need(np.max(np.abs(Jd - Jdo)) <= 1e-10 * np.max(np.abs(Jdo)), "relative DP J")
    ok = not fails
    if fails:
        print("[shared host results] rank %d: %s" % (rank, "; ".join(fails)), flush=True)
    if rank == 0:
        print("[shared host results] %d of 5 kept sweeps in shared slots, values intact, recycled afterwards: %s"
              % (shared, "OK" if ok else "FAILED"), flush=True)
    return bool(ok)


def check_bench_grid(sdp, wl, rank, n_check=300):
    """the bench workload itself (config #5, 2000 x 500 states x <= 256 controls x 9 nodes) on all
    ranks, cut into rows and into columns: value_iteration from a random J and the device-resident
    loop, `n_check` seeded random states against the oracle port (stodynprog.py:639-691)"""
    from oracle.ref_port import port_api
    ora = wl.storage_ar1_large(port_api()).solver
    dims = ora._state_grid_shape
    n_grid = int(np.prod(dims))
    J0 = np.random.default_rng(11).standard_normal(dims)
    picks = np.random.default_rng(12).choice(n_grid, size=n_check, replace=False)
    want_J = np.empty(n_check)
    want_pol = np.empty((n_check, 2))
    if rank == 0:
        Ji = ora.interp_on_state(J0)
        for n, flat in enumerate(picks):
            idx = np.unravel_index(flat, dims)
            x_k = tuple(g[i] for g, i in zip(ora.state_grid, idx))
            want_J[n], want_pol[n] = ora.value_at_state(x_k, Ji)
    ok = True
    for axis in ("rows", "columns"):
        sv = wl.storage_ar1_large(sdp).solver
        sv.slab_axis = axis
        J, pol = sv.value_iteration(J0, report_time=False)
        Js, pols, info = sv.solve_value_iteration(J_zero=J0, max_iter=1)
        T = sv.last_tables
        ok &= T.column and (T.col_bounds is not None) == (axis == "columns")
        if rank == 0:
            for label, Jx, px in (("value_iteration", J, pol), ("solve_value_iteration", Js, pols)):
                bad = int(np.any(px.reshape(n_grid, 2)[picks] != want_pol, axis=1).sum())
                err = float(np.max(np.abs(Jx.reshape(-1)[picks] - want_J) / np.maximum(np.abs(want_J), 1e-300)))
                ok &= bad == 0 and err <= 1e-10
                print("[bench grid 2000x500, %s, shards of %s] %d sampled states: policy mismatches %d, "
                      "J rel err %.2e" % (label, axis, n_check, bad, err), flush=True)
        del sv, T
        torch.cuda.empty_cache()
    return bool(ok)


def main():
    os.environ.setdefault("SDP_P2P_TIMEOUT_S", "120")
    rank = int(os.environ["RANK"])
    local = int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import stodynprog_b200 as sdp
    import workloads as wl
    from conftest import golden, rel_err
    G = golden("storage_ar1.npz")
    layouts = ["control_minor", "state_minor"]
    ok = True
    for layout in layouts:
        prob = wl.storage_ar1(sdp)
        sv = prob.solver
        sv.table_layout = layout
        if layout == "state_minor":
            # force the measured re-cut of the slabs (tolerance 0: any difference moves them)
            from stodynprog_b200.engine import Engine
            Engine.REBALANCE_TOLERANCE = 0.0
            Engine.REBALANCE_SKEW = [1.0 + 0.25 * (r % 2) for r in range(dist.get_world_size())]
            sv.slab_balance = "measured"
        J = prob.J0
        for k in range(3):
            J, pol = sv.value_iteration(J, report_time=False)
            bad = int(np.any(pol != G["vi_pol%d" % k], axis=-1).sum())
            err = rel_err(J, G["vi_J%d" % k])
            ok &= bad == 0 and err <= 1e-10
            if rank == 0:
                print("[%s] sweep %d: policy mismatches %d, J rel err %.2e" % (layout, k, bad, err))
        T = sv.last_tables
        px = sv.engine.peer_exchange(T.host_full.lo.shape[0])
        if rank == 0:
            print("[%s] tables %s, exchange: %s" % (layout, T.layout_name,
                  "peer memory (fused combine + all-gather)" if px is not None else "NCCL all-gather"))
        print("[%s] rank %d slab [%d, %d) backups %d of %d; re-cut: %s" % (
              layout, rank, T.state_begin, T.state_begin + T.n_states, T.n_backups_local,
              T.n_backups_total, T.slab_recut), flush=True)
        if layout == "state_minor":
            ok &= bool(T.slab_recut)
        (Jd, Jr), polp = sv.policy_iteration(prob.initial_policy(), 50, 4, rel_dp=True)
        bad = int(np.any(polp != G["pi_pol"], axis=-1).sum())
        errJ = float(np.max(np.abs(Jd - G["pi_J"])) / np.max(np.abs(G["pi_J"])))
        errR = abs(Jr - float(G["pi_Jref"])) / abs(float(G["pi_Jref"]))
        ok &= bad == 0 and errJ <= 1e-10 and errR <= 1e-10
        if rank == 0:
            print("[%s] policy_iteration: policy mismatches %d, J err %.2e, J_ref %.10g (err %.2e)"
                  % (layout, bad, errJ, Jr, errR))
        # results on rank 0 only: the other ranks pass / receive None
        sv.host_results = "root"
        Jr = prob.J0 if rank == 0 else None
        for k in range(3):
            Jr, polr = sv.value_iteration(Jr, report_time=False)
            if rank == 0:
                ok &= int(np.any(polr != G["vi_pol%d" % k], axis=-1).sum()) == 0
                ok &= rel_err(Jr, G["vi_J%d" % k]) <= 1e-10
            else:
                ok &= Jr is None and polr is None
        Jsr, polsr, infor = sv.solve_value_iteration(J_zero=prob.J0 if rank == 0 else None, max_iter=3, tol=0.0)
        if rank == 0:
            ok &= rel_err(Jsr, G["vi_J2"]) <= 1e-10
            print("[%s] host_results='root': parity on rank 0, None elsewhere" % layout)
        else:
            ok &= Jsr is None
        sv.host_results = "all"
        Js, pols, info = sv.solve_value_iteration(max_iter=3, tol=0.0)
        r_expected = np.max(np.abs(G["vi_J2"] - G["vi_J1"]))
        ok &= rel_err(Js, G["vi_J2"]) <= 1e-10 and abs(info["residuals"][-1] - r_expected) <= 1e-9 * r_expected
    ok &= check_column_layout(sdp, wl, rank)
    ok &= check_shared_results(sdp, wl, rank)
    ok &= check_tiny_grid_and_late_peer(sdp, wl, rank)
    if os.environ.get("SDP_CHECK_BENCH_GRID"):
        ok &= check_bench_grid(sdp, wl, rank)
    flag = torch.tensor([1 if ok else 0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("MULTI_GPU_PARITY", "OK" if flag.item() == 1 else "FAILED")
    dist.destroy_process_group()
    sys.exit(0 if flag.item() == 1 else 1)


if __name__ == "__main__":
    main()
