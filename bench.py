#!/usr/bin/env python
"""bench.py - Bellman backups/s of the sweep hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload large|ar1|pv]
                    [--dump-outputs DIR]

A "step" is one full Bellman sweep (value_iteration's hot path) over the
configured state grid.  Workload: BASELINE.json configs[4], the storage-AR1
problem scaled to 2000 x 500 states x <=256 controls x 9 perturbation nodes
(1 848 240 000 admissible backups per sweep, 38.6 GB of dense tables), sharded over
the N GPUs (strong scaling: total work fixed).  One JSON line on stdout.

  value      whole-job backups/s of a device-resident value iteration, tables and J in
             HBM, CUDA events on the launching stream, barrier + synchronize on both sides,
             max over ranks
  e2e        the same metric through the public API with HOST arrays:
             DPSolver.value_iteration(J_host) -> (J_host, pol_host)
  verified   parity of THIS run, outside the timed regions: 1 000 seeded random states of one
             more sweep - through the timed device path and through value_iteration - against
             the oracle port of the reference's per-state loop
  roofline   a utilisation of the unit that bounds the streaming kernel (named by the library,
             sdp_last_kernel): shared-memory bytes over 128 B/clk/SM for layout CF, streamed /
             algorithmic table bytes over the measured HBM bandwidth otherwise; the dense-
             equivalent rate of SURVEY.md 8d is reported beside it as `dense_equivalent`
  cpu_baseline  the oracle port of the reference's numpy/Cython loop, 1 core (the
             reference is single-threaded), on a bounded random sample of states

--impl reference times the UNMODIFIED reference's own per-state backup
(stodynprog.DPSolver._value_at_state_vect, from the verbatim copy staged under the git-ignored
oracle/_ref/py with its Cython routine compiled from its own source) on bounded samples of the
same workload, 1 core, and prints the same line (kind "reference"; the oracle port when the
staged copy is absent).
--workload pv: BASELINE configs[1], the time-dependent recursion (see run_pv).
--dump-outputs DIR: after the timed steps, what the timed path computed in its last step is
written as DIR/<name>.npy (float64), so that two builds can be compared output for output on
the same seeded inputs (see write_outputs).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

# the benchmark runs from a tree that may be read-only and leaves nothing in it
sys.dont_write_bytecode = True

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
if os.path.join(ROOT, "tests") not in sys.path:
    sys.path.insert(0, os.path.join(ROOT, "tests"))      # workloads.py: the benchmark problem definitions

METRIC = "bellman_backups_per_sec"
UNIT = "backups/s"


def read_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons during the timed region"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.proc = None
        self.lines = []
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": float(max(smax)) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def workload_config(name, dims, W):
    """the `config` object: the workload, stated identically by both arms"""
    return {"workload": name, "states": int(np.prod(dims)), "state_dims": [int(n) for n in dims],
            "perturbation_nodes": int(W),
            "J_init": "default_rng(0).standard_normal on the grid",
            "l2": "GPU arm: every sweep streams its shard of the tables once (4.3 GB on one GPU, "
                  "0.54 GB per GPU on eight; 126 MB of L2), so nothing is flushed between timed "
                  "sweeps; CPU arm: not applicable"}


DUMP_LIMIT_BYTES = 60 * 10 ** 6        # under 64 MB in all, .npy headers included


def write_outputs(out_dir, arrays, seed=0):
    """--dump-outputs: each of `arrays` (name -> array) as out_dir/<name>.npy in float64.
    Above DUMP_LIMIT_BYTES in all, every array keeps the same rows (leading axis) of one
    sample seeded by `seed`, in ascending order."""
    arrays = {k: np.asarray(a, dtype=np.float64) for k, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        n = len(next(iter(arrays.values())))
        rows = np.sort(np.random.default_rng(seed).choice(
            n, size=n * DUMP_LIMIT_BYTES // total, replace=False))
        arrays = {k: a[rows] for k, a in arrays.items()}
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def last_sweep_results(eng, T, J_out):
    """host (J, pol) of the last sweep over the tables T, whose J is the device array J_out:
    one row per state in the grid's C order, as value_iteration returns them.  T holds that
    sweep's argmin until the next sweep over T; K3 maps it to control values."""
    return eng.to_host(J_out, eng.policy_values(T, eng.gather_argmin(T)))


def make_problem(api, args, **solver_kw):
    import workloads as wl
    if args.workload == "ar1":
        return wl.storage_ar1(api, **solver_kw), "howto storage-AR1 41x61 (BASELINE configs[2])"
    prob = wl.storage_ar1_large(api, n_E=args.n_E, n_P=args.n_P, **solver_kw)
    name = "synthetic storage-AR1 %dx%d states x <=256 controls x 9 nodes (BASELINE configs[4])" \
        % (args.n_E, args.n_P)
    return prob, name


def cpu_port_sample(args, n_states, seed=0, interp="c", J=None):
    """time the oracle port's per-state backup (what the reference's value_iteration
    does for each state, stodynprog.py:511-515) on `n_states` random states of the
    workload.  Returns (backups, seconds)."""
    from oracle.ref_port import port_api
    prob, _ = make_problem(port_api(interp), args)
    sv = prob.solver
    dims = sv._state_grid_shape
    rng = np.random.default_rng(seed)
    if J is None:
        J = np.random.default_rng(0).standard_normal(dims)
    J_interp = sv.interp_on_state(J)
    n_grid = int(np.prod(dims))
    picks = rng.choice(n_grid, size=min(n_states, n_grid), replace=False)
    W = len(sv.perturb_grid[0])
    backups = 0
    t0 = time.perf_counter()
    for flat in picks:
        idx = np.unravel_index(flat, dims)
        x_k = tuple(g[i] for g, i in zip(sv.state_grid, idx))
        _, _, _, Jall = sv.value_at_state(x_k, J_interp, None, True)
        backups += Jall.size * W
    return backups, time.perf_counter() - t0


def port_sample_check(args, J_in, results, n_states, seed=1234):
    """Parity of this run's own results, outside the timed region: `n_states` seeded random
    states of the workload's grid are backed up by the oracle port (the reference's per-state
    loop, stodynprog.py:639-691) from the same J_in, and compared with every (label, J_out,
    pol) in `results`.  Returns the `verified` object of the bench line."""
    from oracle import build as ob
    ob.build()
    from oracle.ref_port import port_api
    prob, _ = make_problem(port_api("c"), args)
    sv = prob.solver
    dims = sv._state_grid_shape
    J_interp = sv.interp_on_state(np.asarray(J_in).reshape(dims))
    n_grid = int(np.prod(dims))
    picks = np.random.default_rng(seed).choice(n_grid, size=min(n_states, n_grid), replace=False)
    out = {"states": int(len(picks)), "policy_mismatch": 0, "J_rel": 0.0, "paths": {},
           "checker": "oracle/ref_port.py (per-state numpy loop of the reference) on seeded random "
                      "states of the same grid, same J_next"}
    want_J = np.empty(len(picks))
    want_pol = np.empty((len(picks), len(sv.sys.control)))
    for n, flat in enumerate(picks):
        idx = np.unravel_index(flat, dims)
        x_k = tuple(g[i] for g, i in zip(sv.state_grid, idx))
        want_J[n], want_pol[n] = sv.value_at_state(x_k, J_interp)
    scale = np.maximum(np.abs(want_J), 1e-300)
    for label, J_out, pol in results:
        got_J = np.asarray(J_out).reshape(-1)[picks]
        got_pol = np.asarray(pol).reshape(n_grid, -1)[picks]
        bad = int(np.any(got_pol != want_pol, axis=1).sum())
        err = float(np.max(np.abs(got_J - want_J) / scale))
        out["paths"][label] = {"policy_mismatch": bad, "J_rel": err}
        out["policy_mismatch"] += bad
        out["J_rel"] = max(out["J_rel"], err)
    out["ok"] = bool(out["policy_mismatch"] == 0 and out["J_rel"] <= 1e-10)
    return out


def reference_sample(args, solver, n_states, seed, J=None):
    """time `n_states` seeded random states of the workload through the per-state backup of
    `solver` - the UNMODIFIED reference's DPSolver._value_at_state_vect (stodynprog.py:639-691,
    what its value_iteration calls for each state, :511-515) or the oracle port's restatement.
    Returns (backups, seconds)."""
    dims = solver._state_grid_shape
    n_grid = int(np.prod(dims))
    if J is None:
        J = np.random.default_rng(0).standard_normal(dims)
    J_interp = solver.interp_on_state(J)
    picks = np.random.default_rng(seed).choice(n_grid, size=min(n_states, n_grid), replace=False)
    W = len(solver.perturb_grid[0])
    stock = hasattr(solver, "_value_at_state_vect")
    states = []
    backups = 0
    for flat in picks:                       # (control counts are taken outside the timed loop)
        idx = np.unravel_index(flat, dims)
        x_k = tuple(g[i] for g, i in zip(solver.state_grid, idx))
        states.append(x_k)
        backups += int(np.prod(solver.control_grids(x_k)[1])) * W
    fn = solver._value_at_state_vect if stock else solver.value_at_state
    t0 = time.perf_counter()
    for x_k in states:
        fn(x_k, J_interp)
    return backups, time.perf_counter() - t0


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on this box's host
    cores, bounded samples, rank 0 only.  The stock package (its .py files staged verbatim under
    the git-ignored oracle/_ref/py by __graft_entry__.build(), its Cython routine compiled from
    its own source into oracle/_ref) when present - kind "reference"; else the oracle port."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import contextlib
    import io
    from oracle import build as ob
    ob.build()
    kind, solver, how = "port", None, None
    try:
        from oracle import build_ref
        build_ref.build()
        build_ref.stage_reference_python()
        from oracle.ref_loader import load_reference
        with contextlib.redirect_stdout(io.StringIO()):
            ref = load_reference()
        if ref is not None:
            prob, name = make_problem(ref, args)
            solver = prob.solver
            kind = "reference"
            how = ("the unmodified reference (stodynprog.DPSolver._value_at_state_vect, "
                   "stodynprog.py:639-691, with its own compiled Cython interpolation)")
    except Exception as e:
        sys.stderr.write("stock reference unavailable (%s: %s); timing the oracle port\n"
                         % (type(e).__name__, e))
        solver = None
    if solver is None:
        from oracle.ref_port import port_api
        prob, name = make_problem(port_api("c"), args)
        solver = prob.solver
        how = "the oracle port of the reference's per-state loop (oracle/ref_port.py + sdp_oracle.c)"
    n_sample = args.cpu_sample
    for _ in range(args.warmup):
        reference_sample(args, solver, max(n_sample // 10, 10), seed=99)
    tot_b, tot_t = 0, 0.0
    for k in range(args.steps):
        b, t = reference_sample(args, solver, n_sample, seed=k)
        tot_b += b
        tot_t += t
    value = tot_b / tot_t
    sample = ("%d seeded random states per step of the same %s grid (a full sweep is %d states, "
              "~200 s on one core) through %s; 1 core: the reference is single-threaded (its prange "
              "is compiled without OpenMP, setup.py:21)"
              % (n_sample, "x".join(str(n) for n in solver._state_grid_shape),
                 int(np.prod(solver._state_grid_shape)), how))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * tot_t / max(args.steps, 1), "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(name, solver._state_grid_shape, len(solver.perturb_grid[0])),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": kind, "sample": sample,
                         "host_cpus": os.cpu_count()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def ncu_capture(kernel, n_states):
    """the committed `ncu --set full` capture of this very kernel instantiation on a shard of this
    very size (profiles/r2_traffic.json), or {}: DRAM bytes per launch and pipe utilisations are
    properties of one (kernel, problem) pair and are attached to nothing else"""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as f:
            entries = json.load(f).get("captures", [])
    except Exception:
        return {}
    base = kernel.split(" [")[0]
    for e in entries:
        if e.get("kernel") == base and int(e.get("n_states", -1)) == int(n_states):
            return dict(e, provenance="committed ncu capture (not measured in this run)")
    return {}


def time_sweeps(eng, T, J_prev, J_new, K, barrier):
    """K timed sweeps, CUDA events on the launching stream around the whole loop and
    around each streaming-kernel launch.  Returns (ms_total, k1_ms array, J_prev, J_new)."""
    import torch
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    start.record()
    for k in range(K):
        # a device-resident iteration: between two sweeps the arrival of the peers' J slabs is
        # awaited by the next sweep's first kernel; the last wait is inside the timed region
        # (the policy of an intermediate sweep is read by nobody: only the last one sends its argmin)
        eng.sweep(T, J_prev, J_new, events=kev[k], defer_wait=True, want_argmin=(k == K - 1))
        J_prev, J_new = J_new, J_prev
    eng.flush_exchange()
    end.record()
    barrier()
    from stodynprog_b200 import _cabi
    return (start.elapsed_time(end), np.array([a.elapsed_time(b) for a, b in kev]), J_prev, J_new,
            _cabi.last_kernel())


SMEM_BYTES_PER_CLK_PER_SM = 128       # B200 shared-memory data path (B300_MICROARCH.md)


def roofline_of(T, kernel, k1_ms, ms_total, K, peak, peak_src, sm_count, sm_mhz):
    """roofline object of the streaming kernel `kernel` (the library's own name for what it
    launched).  `frac` is a UTILISATION of the unit that bounds the kernel:
      dense tables (layouts A / B)   HBM: the 4 + 8d + 8/W algorithmic bytes per backup (= what the
                                     kernel streams) over the measured copy bandwidth
      factored tables (AF / BF)      HBM, on the bytes of the compressed tables (each read once per
                                     sweep); the dense-equivalent rate is reported beside it
      layout CF                      shared memory: 16 B per backup (two 8-byte reads of the column
                                     table) over 128 B/clk/SM x SMs x the SM clock of this run
    """
    b_alg = T.algorithmic_bytes_per_backup
    k1 = float(np.mean(k1_ms))
    dense_rate = T.n_backups_local * b_alg / (k1 * 1e-3) / 1e9
    streamed_rate = T.device_bytes / (k1 * 1e-3) / 1e9
    cap = ncu_capture(kernel, T.n_states)
    r = {"kernel": kernel, "kernel_ms": k1, "kernel_share_of_step": k1 * K / ms_total,
         "table_layout": T.layout_name, "table_bytes_resident": T.device_bytes,
         "traffic": cap.get("traffic")}
    hbm = {"achieved": streamed_rate, "peak": peak, "unit": "GB/s", "frac": streamed_rate / peak,
           "peak_source": peak_src, "bytes_per_backup": T.streamed_bytes_per_backup,
           "what": "bytes of table the kernel reads per sweep (each once) / kernel time"}
    if T.column:
        smem_peak = SMEM_BYTES_PER_CLK_PER_SM * sm_count * sm_mhz * 1e6 / 1e9
        smem_rate = T.n_backups_local * 16.0 / (k1 * 1e-3) / 1e9
        r.update({"bound": "smem", "achieved": smem_rate, "peak": smem_peak, "unit": "GB/s",
                  "frac": smem_rate / smem_peak,
                  "peak_source": "%d B/clk/SM x %d SMs x %.0f MHz (SM clock sampled in this run)"
                                 % (SMEM_BYTES_PER_CLK_PER_SM, sm_count, sm_mhz),
                  "algorithmic_bytes_per_backup": 16.0,
                  "algorithmic_bytes_per_launch": T.n_backups_local * 16.0,
                  "hbm": hbm})
    else:
        r.update({"bound": "hbm", "achieved": streamed_rate, "peak": peak, "unit": "GB/s",
                  "frac": streamed_rate / peak, "peak_source": peak_src,
                  "algorithmic_bytes_per_backup": T.streamed_bytes_per_backup if T.factored else b_alg,
                  "algorithmic_bytes_per_launch": float(T.device_bytes) if T.factored
                  else T.n_backups_local * b_alg})
        if not T.factored:
            # (padding of the dense layouts counts against the fraction: streamed >= algorithmic)
            r["achieved"] = dense_rate
            r["frac"] = dense_rate / peak
            r["padding_fill"] = T.n_backups_local / max(T.n_entries, 1)
            r["streamed_GBs"] = streamed_rate
    if T.factored:
        r["dense_equivalent"] = {
            "achieved": dense_rate, "unit": "GB/s", "over_hbm_peak": dense_rate / peak,
            "bytes_per_backup": b_alg,
            "what": "SURVEY.md 8d figure: the dense (x,u,w) layout's 4 + 8d + 8/W bytes per backup x "
                    "backups / kernel time - NOT a utilisation: the compressed tables never stream "
                    "those bytes (see `dense_layout` for the kernel that does)"}
    if cap:
        r["ncu"] = {k: v for k, v in cap.items() if k not in ("traffic", "kernel", "n_states")}
    return r


def run_ours(args):
    # a rank that dies must fail the run quickly, not leave its peers spinning on flags
    os.environ.setdefault("SDP_P2P_TIMEOUT_S", "120")
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); "
                         "use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    import stodynprog_b200 as sdp
    from stodynprog_b200 import _cabi
    from stodynprog_b200 import build as product_build
    if rank == 0:
        product_build.build()
    if world > 1:
        dist.barrier()

    prob, name = make_problem(sdp, args)
    sv = prob.solver
    if args.layout != "auto":
        sv.table_layout = args.layout
    sv.table_compress = args.compress
    sv.column_hoist = args.column_hoist
    if args.item_chunk:
        sv._item_chunk = args.item_chunk
    # table build: dyn/cost evaluated chunk by chunk on several host threads (DPSolver.host_threads,
    # an opt-in: the reference calls them on the calling thread); the box's cores shared by the ranks
    ncpu = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    sv.host_threads = max(1, min(16, ncpu // world)) if args.host_threads == "auto" else int(args.host_threads)
    eng = sv.engine
    t0 = time.perf_counter()
    T = sv.sweep_tables()
    setup_s = time.perf_counter() - t0
    dims = sv._state_grid_shape
    n_grid = int(np.prod(dims))

    J_host = np.random.default_rng(0).standard_normal(dims)
    J_prev, J_new = eng.J_pair(n_grid)
    eng.begin_call(n_grid)
    eng.upload_J(J_host, J_prev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # clocks / throttle reasons are sampled from the warm-up to the end of the e2e loop
    # (the device-timed region alone is only K x 3 ms: too short for nvidia-smi's 100 ms period)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.2)
    for _ in range(args.warmup):
        eng.sweep(T, J_prev, J_new, defer_wait=True)
        J_prev, J_new = J_new, J_prev
    eng.flush_exchange()

    K = args.steps
    launches0 = _cabi.launch_count()
    ms_total, k1_ms, J_prev, J_new, kernel = time_sweeps(eng, T, J_prev, J_new, K, barrier)
    launches = _cabi.launch_count() - launches0
    t = torch.tensor([ms_total, float(np.mean(k1_ms))], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total_max, k1_ms_max = float(t[0]), float(t[1])
    k1_per_rank = None
    if world > 1:
        # slab balance: every rank's mean streaming-kernel time and slab size
        mine = torch.tensor([float(np.mean(k1_ms)), float(T.n_backups_local), float(T.n_states)],
                            dtype=torch.float64, device="cuda")
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        k1_per_rank = {"balance": "re-cut by measured slab times" if T.slab_recut else "equal admissible controls",
                       "kernel_ms_before_recut": T.slab_times_ms,
                       "kernel_ms": [round(float(x[0]), 4) for x in allr],
                       "backups": [int(x[1]) for x in allr], "states": [int(x[2]) for x in allr]}
    total_backups = T.n_backups_total
    value = total_backups * K / (ms_total_max * 1e-3)

    peak, peak_src = read_peaks()
    J_keep = J_prev.clone()
    if args.dump_outputs:
        # (before the e2e calls below sweep over T again)
        J_last, pol_last = last_sweep_results(eng, T, J_keep)
        if rank == 0:
            write_outputs(args.dump_outputs, {"J": J_last.reshape(n_grid),
                                              "pol": pol_last.reshape(n_grid, -1)})
        del J_last, pol_last

    # end-to-end through the public API, host arrays in and out
    n_e2e = max(3, min(K, 10))

    def time_e2e(mode):
        """n_e2e calls of value_iteration with host arrays; `mode` = solver.host_results"""
        sv.host_results = mode
        J_h = J_keep.cpu().numpy().reshape(dims)
        for _ in range(2):
            J_h, pol_h = sv.value_iteration(J_h, report_time=False)
        barrier()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            J_h, pol_h = sv.value_iteration(J_h, report_time=False)
        torch.cuda.synchronize()
        e2e_local = time.perf_counter() - t0
        te = torch.tensor([e2e_local], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e_s = float(te[0])
        if rank == 0 and os.environ.get("SDP_SHARED_TIMING") and getattr(eng, "last_shared_timing", None):
            sys.stderr.write("shared-results call, host ms per stage [slots, upload, sweep, results, cache check, "
                             "gpu wait, barrier]: %s\n" % ["%.3f" % (1e3 * x) for x in eng.last_shared_timing])
        nb_J = 8 * n_grid
        nb_pol = 8 * n_grid * len(sv.sys.control)
        copying = world if mode == "all" else 1       # ranks that move host data
        return {"value": total_backups * n_e2e / e2e_s, "unit": UNIT,
                "h2d_bytes_per_step": nb_J * copying, "d2h_bytes_per_step": (nb_J + nb_pol) * copying,
                "steps": n_e2e, "ms_per_step": 1e3 * e2e_s / n_e2e,
                "api": "DPSolver.value_iteration(J_host) -> (J_host, pol_host)" + (
                    "" if world == 1 else
                    ", solver.host_results = 'all': every rank uploads J and downloads (J, pol)" if mode == "all"
                    else ", solver.host_results = 'root': rank 0 uploads J (handed to the other ranks "
                         "over NVLink) and rank 0 alone downloads (J, pol)")}

    e2e = time_e2e("all")
    clocks = sampler.stop() if rank == 0 else None
    # roofline of the streaming kernel on this rank's shard (rank 0's is printed)
    props = torch.cuda.get_device_properties(local_rank)
    sm_count = props.multi_processor_count
    sm_mhz = (clocks or {}).get("sm_mhz") or getattr(props, "clock_rate", 1965000) / 1e3
    roofline = roofline_of(T, kernel, k1_ms, ms_total, K, peak, peak_src, sm_count, sm_mhz)
    e2e_all = None
    if world > 1:
        # 8 ranks pulling 24 MB each through shared PCIe roots take ~2 ms, one rank 0.45 ms
        # (scripts/dev_pcie_contention.py): the headline uses the root-only result mode
        e2e_all = e2e
        e2e = time_e2e("root")
        sv.host_results = "all"

    # parity of THIS run, outside the timed regions: one more sweep from J_keep through the
    # device-resident path that was timed (Engine.sweep + exchange) and one through the public
    # API (the e2e path), both compared with the oracle port on seeded random states
    verified = None
    if args.verify_states > 0:
        Ja, Jb = eng.J_pair(n_grid)
        eng.begin_call(n_grid)
        Ja.copy_(J_keep)
        eng.sweep(T, Ja, Jb)
        pol_dev = eng.policy_values(T, eng.gather_argmin(T))
        J_dev_out, pol_dev_out = eng.to_host(Jb, pol_dev)
        J_in_host = J_keep.cpu().numpy().reshape(dims)
        sv.host_results = "all"
        J_api_out, pol_api_out = sv.value_iteration(J_in_host.copy(), report_time=False)
        if rank == 0:
            verified = port_sample_check(args, J_in_host, [
                ("Engine.sweep (device-resident, timed path)", J_dev_out, pol_dev_out),
                ("DPSolver.value_iteration (e2e path)", J_api_out, pol_api_out)], args.verify_states)
        barrier()

    # the same workload through the dense (x,u,w) tables: the HBM-bound kernel the
    # roofline target is stated for (SURVEY.md 8d)
    dense = None
    if T.factored and not args.no_dense:
        sv.table_compress = "off"
        sv.column_hoist = "off"
        Td = sv.sweep_tables()
        Ja, Jb = eng.J_pair(n_grid)
        eng.begin_call(n_grid)
        Ja.copy_(J_keep)
        for _ in range(3):
            eng.sweep(Td, Ja, Jb)
            Ja, Jb = Jb, Ja
        Kd = max(5, min(K, 10))
        ms_d, k1_d, Ja, Jb, kernel_d = time_sweeps(eng, Td, Ja, Jb, Kd, barrier)
        td = torch.tensor([ms_d], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(td, op=dist.ReduceOp.MAX)
        dense = {"value": total_backups * Kd / (float(td[0]) * 1e-3), "unit": UNIT, "steps": Kd,
                 "ms_per_step": float(td[0]) / Kd,
                 "roofline": roofline_of(Td, kernel_d, k1_d, ms_d, Kd, peak, peak_src, sm_count, sm_mhz)}
        sv.table_compress = args.compress
        sv.column_hoist = args.column_hoist
        del Td
        sv.clear_tables()
        torch.cuda.empty_cache()

    setup = torch.tensor([setup_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(setup, op=dist.ReduceOp.MAX)

    extra = None
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import build as ob
        ob.build()
        b, tcpu = cpu_port_sample(args, args.cpu_sample, seed=0)
        cpu = {"value": b / tcpu, "unit": UNIT, "cores": 1, "kind": "port",
               "host_cpus": os.cpu_count(), "seconds": tcpu,
               "sample": "%d random states (seeded) of the same grid, %d backups, per-state "
                         "numpy loop of the reference restated in oracle/ref_port.py (the "
                         "reference is single-threaded: prange compiled without OpenMP)"
                         % (args.cpu_sample, b)}
    if rank == 0 and world == 1 and args.workload == "large" and not args.no_extra:
        extra = measure_config3(sdp, peak, peak_src, sm_count, sm_mhz)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K,
            "warmup": args.warmup, "ms_per_step": ms_total_max / K, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(name, dims, T.W),
            "plan": {"backups_per_sweep": total_backups, "table_layout": T.layout_name,
                     "row_bands": (T.bands["rows"] if T.column else None),
                     # (the e2e path sweeps the columns in pieces, each on its way to the host
                     # while the next ones are swept)
                     "column_pieces": ([[ch["c0"], ch["c1"]] for ch in eng._chunk_plan(T)]
                                       if (T.column and world == 1 and eng.can_overlap_results(T)
                                           and len(T.bands["tiles"]) == 1) else None),
                     "shard_axis": (None if world == 1 else "columns" if T.col_bounds is not None else "rows"),
                     "tabulate_mode": T.tabulate_mode, "host_threads": int(sv.host_threads),
                     "item_chunk": T.item_chunk,
                     "table_gb_per_gpu": T.device_bytes / 1e9,
                     "parallelism": "state shards x%d, %s" % (
                         world, "one rank" if world == 1 else
                         ("J shard stored into every rank's buffer by the combine kernel over NVLink "
                          "peer memory + flag wait" if eng.peer_exchange(n_grid) is not None
                          else "NCCL all-gather of J per sweep"))},
            "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline,
            "clocks": clocks, "setup_seconds": float(setup[0]),
            # rank 0's build, seconds per stage: scan of the control boxes, layout decisions,
            # dyn/cost evaluation + staging copies + uploads + K0 launches (pipelined), work list,
            # and the wait for the device work still in flight at the end
            "setup_split": T.setup_split,
        }
        if verified is not None:
            line["verified"] = verified
        if e2e_all is not None:
            line["e2e_all_ranks"] = e2e_all
        if k1_per_rank is not None:
            line["slabs"] = k1_per_rank
        if dense is not None:
            line["dense_layout"] = dense
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if extra is not None:
            line["storage_ar1_41x61"] = extra
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_pv(args):
    """--workload pv: BASELINE configs[1], the time-dependent deterministic storage problem
    (examples/01 .../pv_storage_control.py: 50 states x 1 001..2 001 controls, T = 240 instants,
    17 894 880 backups per recursion).  A step = one whole bellman_recursion(T, J_fin).
      value  backups/s of the recursion proper: tables of all instants resident, the T sweeps
             enqueued back to back, one copy of (J, pol) to the host (Engine.recursion_fast)
      e2e    backups/s of the public call DPSolver.bellman_recursion(T, J_fin) -> (J, pol),
             INCLUDING the host tabulation of the user's callables for all instants
      cpu_baseline  the same recursion through the oracle port / the stock reference, 1 core"""
    import contextlib
    import io
    import torch
    import stodynprog_b200 as sdp
    import workloads as wl
    from stodynprog_b200 import _cabi
    from stodynprog_b200 import build as product_build
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(0)
    product_build.build()
    prob = wl.pv_storage(sdp)
    sv = prob.solver
    name = "examples/01 deterministic PV storage: 50 states x 1001..2001 controls x T=240 (BASELINE configs[1])"
    quiet = contextlib.redirect_stdout(io.StringIO())
    for _ in range(max(args.warmup, 1)):
        with quiet:
            J, pol = sv.bellman_recursion(prob.horizon, prob.J_fin)
    backups = sv.last_tables.n_backups_total * prob.horizon
    launches0 = _cabi.launch_count()
    walls, sweeps, tabs = [], [], []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        with quiet:
            J, pol = sv.bellman_recursion(prob.horizon, prob.J_fin)
        walls.append(time.perf_counter() - t0)
        info = sv.last_recursion or {}
        sweeps.append(info.get("sweeps_s", float("nan")))
        tabs.append(info.get("tabulate_s", float("nan")) + info.get("upload_build_s", float("nan")))
    launches = _cabi.launch_count() - launches0
    if args.dump_outputs:
        write_outputs(args.dump_outputs, {"J": J, "pol": pol})
    from oracle import build as ob
    ob.build()
    from oracle.ref_port import port_api
    ora = wl.pv_storage(port_api())
    t0 = time.perf_counter()
    Jo, polo = ora.solver.bellman_recursion(ora.horizon, ora.J_fin)
    t_cpu = time.perf_counter() - t0
    bad = int(np.any(pol != polo, axis=-1).sum())
    err = float(np.max(np.abs(J - Jo) / np.maximum(np.abs(Jo), 1e-300)))
    line = {
        "metric": METRIC, "value": backups / float(np.mean(sweeps)), "unit": UNIT, "n_gpus": 1,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * float(np.mean(sweeps)),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": name, "states": 50, "instants": int(prob.horizon), "backups_per_recursion": backups},
        "e2e": {"value": backups / float(np.mean(walls)), "unit": UNIT, "ms_per_step": 1e3 * float(np.mean(walls)),
                "h2d_bytes_per_step": int(8 * (sv.last_tables.g.numel() * prob.horizon + 50)),
                "d2h_bytes_per_step": int(8 * 2 * 50 * prob.horizon),
                "api": "DPSolver.bellman_recursion(T, J_fin) -> (J, pol), user callables tabulated inside",
                "tabulate_upload_ms": 1e3 * float(np.mean(tabs)), "sweeps_and_copy_ms": 1e3 * float(np.mean(sweeps))},
        "gpu_launches": int(launches), "recursion_path": "fast" if sv.last_recursion else "per_instant",
        "verified": {"states": int(Jo.size), "policy_mismatch": bad, "J_rel": err, "ok": bool(bad == 0 and err <= 1e-10),
                     "checker": "oracle/ref_port.py, the whole recursion"},
        "cpu_baseline": {"value": backups / t_cpu, "unit": UNIT, "cores": 1, "kind": "port", "seconds": t_cpu,
                         "sample": "the whole T=240 recursion through oracle/ref_port.py"},
    }
    print(json.dumps(line))


def measure_config3(sdp, peak, peak_src, sm_count, sm_mhz, steps=50, warmup=5):
    """BASELINE configs[2] (the 41x61 storage-AR1 grid of the notebook, 142 762 509
    backups per sweep): the grid the north star's 60 % roofline target is quoted on.
    Reported for the default (factored) tables and for the dense tables."""
    import torch
    import workloads as wl
    out = {"workload": "howto storage-AR1 41x61 x 4001..8001 controls x 9 nodes"}
    for compress in ("auto", "off"):
        prob = wl.storage_ar1(sdp)
        sv = prob.solver
        sv.table_compress = compress
        eng = sv.engine
        T = sv.sweep_tables()
        J_prev, J_new = eng.J_pair(41 * 61)
        eng.upload_J(np.random.default_rng(0).standard_normal(41 * 61), J_prev)
        for _ in range(warmup):
            eng.sweep(T, J_prev, J_new)
            J_prev, J_new = J_new, J_prev
        ms_total, k1_ms, J_prev, J_new, kernel = time_sweeps(eng, T, J_prev, J_new, steps,
                                                             torch.cuda.synchronize)
        out["backups_per_sweep"] = T.n_backups_total
        out["default" if compress == "auto" else "dense_layout"] = {
            "ms_per_step": ms_total / steps, "value": T.n_backups_total * steps / (ms_total * 1e-3),
            "unit": UNIT,
            "roofline": roofline_of(T, kernel, k1_ms, ms_total, steps, peak, peak_src, sm_count, sm_mhz)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="large", choices=["large", "ar1", "pv"])
    ap.add_argument("--n-E", dest="n_E", type=int, default=2000)
    ap.add_argument("--n-P", dest="n_P", type=int, default=500)
    ap.add_argument("--layout", default="auto", choices=["auto", "control_minor", "state_minor"])
    ap.add_argument("--compress", default="auto", choices=["auto", "off", "on"],
                    help="factored (x,u)+(x,w) tables (auto: whenever the system allows)")
    ap.add_argument("--column-hoist", dest="column_hoist", default="auto", choices=["auto", "on", "off"],
                    help="layout CF, one inner-interpolation table per grid column (auto: SDP_COLUMN_HOIST)")
    ap.add_argument("--host-threads", dest="host_threads", default="auto",
                    help="host threads of the table build (auto = cores / ranks, at most 16; 1 = calling thread only)")
    ap.add_argument("--no-dense", action="store_true", help="skip the dense-layout sub-measurement")
    ap.add_argument("--item-chunk", dest="item_chunk", type=int, default=0)
    ap.add_argument("--cpu-sample", dest="cpu_sample", type=int, default=None,
                    help="states per CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--verify-states", dest="verify_states", type=int, default=1000,
                    help="states of the final sweep checked against the oracle port (0: skip)")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR", default=None,
                    help="write the timed path's results of its last step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm times samples of states, not whole results")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.cpu_sample is None:
        # ~200 us per state for the 2000x500 grid (<=256 controls); ~1.4 ms for the 41x61 grid
        args.cpu_sample = (60000 if args.impl == "ours" else 8000) if args.workload == "large" else 2501
    if args.workload == "pv" and args.impl == "ours":
        run_pv(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
