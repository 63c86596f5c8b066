"""DPSolver - the reference's solver API on top of the B200 sweep engine.

Drop-in for `stodynprog.DPSolver` (reference stodynprog/stodynprog.py:317-876):
same constructor, attributes (`state_grid`, `perturb_grid`, `perturb_proba`,
`control_steps`, `_state_grid_shape`, `_state_ref_ind`, `_state_ref`), methods,
argument meaning, return conventions (host numpy fp64 arrays; policies hold
control VALUES), printed progress lines and error behaviour.  What changes is
where the loop nest runs:

  reference                                     here
  ---------                                     ----
  Python loop over states (:511-515)            one K1 launch over the slab
  per-state dyn/cost callbacks (:674-676)       tabulated once per (sys, grids),
                                                tables resident in HBM
  Cython cell search + lerp (pyx:54-300)        K0 (cell search) + K1 (gather/lerp)
  np.inner over w, argmin over u (:682-686)     registers + warp shuffles in K1
  eval_policy iteration (:743-763)              K1' launches, J stays on the device

The constructor accepts two optional keyword arguments the reference does not
have: `device` and `group` (a torch.distributed process group) to shard the
state grid over the GPUs of one box.
"""
import itertools
from datetime import datetime

import os

import numpy as np

from . import tabulate as tb
from .interp import MlinInterpolator

__all__ = ["DPSolver"]


class DPSolver(object):
    def __init__(self, sys, device=None, group=None, cache_tables=True, item_chunk=None,
                 _test_lib=None):
        """Dynamic Programming solver for the stochastic control of `sys`
        (a `SysDescription`).  Implements Value Iteration, Policy Iteration
        (policy evaluation by repeated fixed-policy backups) and the
        finite-horizon Bellman recursion.  (reference stodynprog.py:318-333)"""
        self.sys = sys
        # default 1-point grids, like the reference (:328-332)
        self.state_grid = [[0.] for s in self.sys.state]
        self.perturb_grid = [[0.] for p in self.sys.perturb]
        self.perturb_proba = [[1.] for p in self.sys.perturb]
        self.control_steps = (1.,) * len(self.sys.control)
        # device side (created lazily: grids can be set up without a GPU)
        self._device = device
        self._group = group
        self._item_chunk = item_chunk
        self._test_lib = _test_lib      # test seam, see Engine.__init__
        self._engine = None
        self.cache_tables = bool(cache_tables)
        self._table_cache = {}
        self.last_tables = None      # SweepTables of the last sweep (bench / diagnostics)
        # table layout and host tabulation mode (see Engine.build_sweep_tables)
        self.table_layout = "auto"    # "auto" | "control_minor" | "state_minor"
        self.tabulate = "auto"        # "auto" | "per_state" | "batched"
        # batched tabulation: host threads that evaluate dyn/cost on chunks of states.  1 (the
        # default, or SDP_HOST_THREADS) calls them on the calling thread only, as the reference does;
        # more is an opt-in for callables that are thread-safe (pure numpy code is): "auto" = the
        # cores this process may run on, at most 16.  Same calls, same tables either way.
        self.host_threads = os.environ.get("SDP_HOST_THREADS", "1")
        # "auto": keep the tables as a (x,u) part + a (x,w) part whenever dyn/cost
        # have that structure (every reference example does); "off": always dense
        self.table_compress = "auto"  # "auto" | "off" | "on"
        # layout CF, column-shared hoist (include/sdp_b200.h): when state axis 0 alone follows
        # the control and the (x,w) part of the next state does not depend on axis 0 (the
        # storage examples), one CTA tabulates the inner interpolation once per column of
        # the grid; "auto" follows SDP_COLUMN_HOIST, "on" raises if it does not apply
        self.column_hoist = "auto"    # "auto" | "on" | "off"
        # layout CF: a lane of the sweep owns two neighbouring rows of a column, whose backups
        # read overlapping rows of the column table (3 shared-memory reads for 2 backups);
        # "auto" follows SDP_COLUMN_PAIRS
        self.column_pairs = "auto"    # "auto" | "on" | "off"
        # several ranks, layout CF: cut the grid into slabs of whole rows of axis 0 ("rows") or
        # into whole columns ("columns": the per-column costs then divide by the number of
        # ranks); "auto" (SDP_SLAB_AXIS) takes columns wherever layout CF applies and every rank
        # gets at least 4 of them
        self.slab_axis = "auto"       # "auto" | "rows" | "columns"
        # several ranks: cut the grid into slabs of equal admissible controls ("controls"), or
        # re-cut once by the measured sweep time of every slab ("measured"; "auto" does so
        # for sweeps of at least 5e8 backups)
        self.slab_balance = "auto"    # "auto" | "controls" | "measured"
        # several ranks: "all" = every rank passes J_next and gets (J_k, pol_k), as an
        # unchanged SPMD script expects; "root" = only rank 0's J_next is read (it is
        # handed to the other ranks over NVLink) and only rank 0 gets host results, the
        # others get None - 8 ranks pulling 24 MB each through a shared PCIe root take
        # 2 ms, one rank 0.45 ms.  value_iteration / solve_value_iteration only.
        self.host_results = "all"     # "all" | "root"
        # bellman_recursion: "auto" tabulates all instants up front and runs the sweeps back to
        # back when only the stage cost depends on the instant; "per_instant" never does
        self.recursion_mode = "auto"  # "auto" | "per_instant"
        self.last_recursion = None    # timings of the last fast recursion (diagnostics)

    # ------------------------------------------------------------------
    # discretisation (host only)
    # ------------------------------------------------------------------
    def discretize_perturb(self, *linspace_args):
        """regular grid + probability weights for each perturbation
        (3 linspace arguments per perturbation; reference stodynprog.py:335-362).
        Continuous laws: pdf on the grid normalised to sum 1; discrete laws: pmf,
        which must already sum to 1."""
        assert len(linspace_args) == len(self.sys.perturb) * 3
        self.perturb_grid = []
        self.perturb_proba = []
        for i in range(len(self.sys.perturb)):
            grid_wi = np.linspace(*linspace_args[i * 3:i * 3 + 3])
            law = self.sys.perturb_laws[i]
            if self.sys.perturb_types[i] == 'continuous':
                proba_wi = law.pdf(grid_wi)
                proba_wi /= proba_wi.sum()
            else:
                proba_wi = law.pmf(grid_wi)
                assert np.allclose(proba_wi.sum(), 1.)
            self.perturb_grid.append(grid_wi)
            self.perturb_proba.append(proba_wi)
        return self.perturb_grid, self.perturb_proba

    def discretize_state(self, *linspace_args):
        """regular grid for each state variable (3 linspace arguments each);
        also records the grid shape and the reference state of relative DP, the
        middle of the grid (reference stodynprog.py:364-389)."""
        assert len(linspace_args) == len(self.sys.state) * 3
        self.state_grid = [np.linspace(*linspace_args[i * 3:i * 3 + 3])
                           for i in range(len(self.sys.state))]
        shape = tuple(len(g) for g in self.state_grid)
        self._state_grid_shape = shape
        self._state_ref_ind = tuple(nx // 2 for nx in shape)
        self._state_ref = tuple(g[i] for g, i in zip(self.state_grid, self._state_ref_ind))
        return self.state_grid

    @property
    def state_grid_full(self):
        """broadcast (meshgrid-like) view of the state grid
        (reference stodynprog.py:391-403)"""
        nd = len(self.state_grid)
        axes = [np.reshape(g, (1,) * i + (-1,) + (1,) * (nd - i - 1))
                for i, g in enumerate(self.state_grid)]
        return np.broadcast_arrays(*axes)

    def interp_on_state(self, A):
        """interpolating function of array `A` given on the state grid
        (reference stodynprog.py:405-430)"""
        expect_shape = self._state_grid_shape
        if A.shape != expect_shape:
            raise ValueError('array `A` should be of shape {:s}, not {:s}'.format(
                str(expect_shape), str(A.shape)))
        if len(expect_shape) <= 5:
            A_interp = MlinInterpolator(*self.state_grid)
            A_interp.set_values(A)
            return A_interp
        raise NotImplementedError('interpolation for state dimension >5'
                                  ' is not implemented.')

    def control_grids(self, state_k, t_k=None):
        """grid of admissible controls at `state_k`: (list of 1-D grids, dims)
        using `control_steps` as step hints (reference stodynprog.py:432-463)"""
        if t_k is not None:
            state_k = (t_k,) + state_k
        intervals = self.sys.control_box(*state_k, **self.sys.params)
        lo, hi, npts = tb.control_grid_counts(intervals, self.control_steps)
        grids = [tb.make_control_grid(a, b, n) for a, b, n in zip(lo, hi, npts)]
        return grids, tuple(npts)

    # ------------------------------------------------------------------
    # device plumbing
    # ------------------------------------------------------------------
    @property
    def engine(self):
        if self._engine is None:
            from .engine import Engine
            self._engine = Engine(self._device, self._group, self._item_chunk, self._test_lib)
        return self._engine

    def _cache_key(self, t_k):
        def sig(a):
            a = np.ascontiguousarray(np.asarray(a, dtype=float))
            return (a.shape, a.tobytes())
        s = self.sys
        return (t_k, id(s.dyn), id(s.cost), id(s.control_box),
                repr(sorted(s.params.items())) if s.params else '',
                tuple(sig(g) for g in self.state_grid),
                tuple(sig(g) for g in self.perturb_grid),
                tuple(sig(p) for p in self.perturb_proba),
                tuple(float(c) for c in self.control_steps),
                self.table_layout, self.tabulate, self.table_compress, self.slab_balance,
                getattr(self, "column_hoist", "auto"), getattr(self, "slab_axis", "auto"),
                getattr(self, "column_pairs", "auto"))

    def clear_tables(self):
        """drop the device-resident tables (call after mutating anything the
        user callables read from their enclosing scope)"""
        self._table_cache = {}
        self.last_tables = None
        if self._engine is not None:
            self._engine._scan_cache = None
            self._engine._grid_cache = {}

    def _probe_fingerprint(self, t_k=None):
        """What the user's control_box / dyn / cost return TODAY on three probe states (first,
        middle, last of the grid), as bytes.  The reference calls them afresh in every sweep
        (stodynprog.py:440,674,676), so callables that read module globals or closure cells - its
        own doc/example_inventory.py cost reads (h, p, c) - see changes made between two calls;
        cached tables are only reused while this fingerprint is unchanged."""
        sys = self.sys
        grids = [np.asarray(g, dtype=float) for g in self.state_grid]
        dims = [len(g) for g in grids]
        w_args, w_shape, W = tb.perturb_layout(self.perturb_grid)
        out = []
        for idx in ([0] * len(dims), [n // 2 for n in dims], [n - 1 for n in dims]):
            x_k = tuple(g[i] for g, i in zip(grids, idx))
            tab = tb.scan_control_boxes(sys, self.control_steps, [x_k], t_k)
            out += [tab.lo.tobytes(), tab.hi.tobytes(), tab.npts.tobytes()]
            compact, _, _ = tb._eval_one_state(sys, x_k, tab, 0, w_args, t_k, W, w_shape)
            out += [a.tobytes() for a, _, _ in compact]
        return b"".join(out)

    def _cached_tables(self, t_k):
        return self._table_cache.get(self._cache_key(t_k)) if self.cache_tables else None

    def _tables_still_valid(self, T, t_k=None):
        """False when the callables no longer give what the cached tables `T` were built from
        (same answer on every rank: the probe states are grid states, not shard states)"""
        fp = getattr(T, "probe_fingerprint", None)
        return fp is None or fp == self._probe_fingerprint(t_k)

    def sweep_tables(self, t_k=None, reuse=None, validate=True):
        """device tables for the current (sys, grids, control_steps[, t_k]); cached stationary
        tables are re-validated against the callables (`_probe_fingerprint`) unless the caller
        does that itself while the GPU works (`_sweep_host`)"""
        if not self.cache_tables:
            T = self.engine.build_sweep_tables(self, t_k, reuse=reuse)
            self.last_tables = T
            return T
        key = self._cache_key(t_k)
        T = self._table_cache.get(key)
        if T is not None and validate and not self._tables_still_valid(T, t_k):
            self.clear_tables()
            T = None
        if T is None:
            T = self.engine.build_sweep_tables(self, t_k, reuse=reuse)
            if t_k is None:
                # stationary tables are reused across sweeps / policy iterations
                T.probe_fingerprint = self._probe_fingerprint(t_k)
                self._table_cache = {key: T}
        self.last_tables = T
        return T

    def _root_only(self):
        if getattr(self, "host_results", "all") not in ("all", "root"):
            raise ValueError("host_results must be 'all' or 'root'")
        return self.host_results == "root" and self.engine.coll.world > 1

    def _sweep_host(self, J_next, t_k=None, rel_dp=False, tables=None):
        """one sweep with host arrays in/out. Returns (J_k, J_ref or None, pol_k, tables)"""
        import torch
        eng = self.engine
        state_dims = tuple(len(g) for g in self.state_grid)
        nb_control = len(self.sys.control)
        # cached tables are launched at once and checked against the callables WHILE the GPU
        # sweeps (the host would only wait); a stale cache costs one wasted sweep, then a rebuild
        cached = tables is None and self._cached_tables(t_k) is not None
        T = tables if tables is not None else self.sweep_tables(t_k, validate=False)
        stale = []

        def check_cache():
            if cached and not stale and not self._tables_still_valid(T, t_k):
                stale.append(True)

        n_grid = int(np.prod(state_dims))
        root_only = self._root_only()
        is_root = eng.coll.rank == 0
        hs = eng.host_share(n_grid, nb_control) if eng.coll.world > 1 else None
        if hs is not None:
            # several ranks: inputs and results through page-locked memory shared by the ranks,
            # 1/N of each over every rank's own PCIe link (hostshare.py)
            ref_flat = int(np.ravel_multi_index(self._state_ref_ind, state_dims)) if rel_dp else None
            got = eng.sweep_shared(hs, T, J_next, rel_ref_index=ref_flat,
                                   want_results=not (root_only and not is_root), while_waiting=check_cache)
            if stale:
                self.clear_tables()
                return self._sweep_host(J_next, t_k, rel_dp)
            if got is not None:
                if got[0] is None:
                    return None, None, None, T
                hs_, slot, J_ref = got
                # rank 0 may write into what it gets (the next call reads ITS array); the other
                # ranks share the same pages and get read-only views
                J_k, pol_k = hs_.hand_out(slot, state_dims, state_dims + (nb_control,), writable=is_root)
                return J_k, J_ref, pol_k, T
        J_prev, J_new = eng.J_pair(n_grid)
        eng.begin_call(n_grid)
        if root_only:
            if is_root:
                eng.upload_J(J_next, J_prev)
            eng.share_J(J_prev)
        else:
            eng.upload_J(J_next, J_prev)
        if not rel_dp and eng.can_overlap_results(T):
            # large single-rank sweep: results stream to the host while later runs compute
            J_k, pol_k = eng.sweep_to_host(T, J_prev, J_new, while_waiting=check_cache)
            if stale:
                self.clear_tables()
                return self._sweep_host(J_next, t_k, rel_dp)
            return J_k.reshape(state_dims), None, pol_k.reshape(state_dims + (nb_control,)), T
        ref_out = None
        ref_flat = None
        if rel_dp:
            ref_flat = int(np.ravel_multi_index(self._state_ref_ind, state_dims))
            ref_out = torch.zeros(1, dtype=torch.float64, device=eng.device)
        eng.sweep(T, J_prev, J_new, rel_ref_index=ref_flat, ref_out=ref_out)
        argmin_full = eng.gather_argmin(T)
        if root_only and not is_root:
            check_cache()
            if stale:
                self.clear_tables()
                return self._sweep_host(J_next, t_k, rel_dp)
            return None, None, None, T           # results travel to rank 0's host only
        pol_dev = eng.policy_values(T, argmin_full)               # K3: indices -> control values
        outs = eng.to_host(J_new, pol_dev, *([ref_out] if rel_dp else []), while_waiting=check_cache)
        if stale:
            self.clear_tables()
            return self._sweep_host(J_next, t_k, rel_dp)
        J_k = outs[0].reshape(state_dims)
        pol_k = outs[1].reshape(state_dims + (nb_control,))
        J_ref = float(outs[2][0]) if rel_dp else None
        return J_k, J_ref, pol_k, T

    # ------------------------------------------------------------------
    # solvers
    # ------------------------------------------------------------------
    def value_iteration(self, J_next, rel_dp=False, report_time=True):
        """solve one DP step on the entire state grid, given the cost-to-go
        array `J_next` on that grid.

        If rel_dp is True, J_next should be a (J_next, J_ref) tuple.

        Returns (J_k, pol_k); J_k is a tuple (J_diff, J_ref) if `rel_dp`.
        (reference stodynprog.py:466-534)
        """
        t_start = datetime.now()
        ref_ind = getattr(self, '_state_ref_ind', None)
        # host_results == "root": the other ranks' J_next is not read (it may be None)
        ignored = self._root_only() and self.engine.coll.rank != 0
        if rel_dp:
            J_next, J_ref = J_next if J_next is not None else (None, None)
            # the cost-to-go must be a *differential* cost, zero at the reference state
            assert ignored or J_next[ref_ind] == 0.
        state_dims = tuple(len(g) for g in self.state_grid)
        if not ignored:
            J_next = np.asarray(J_next)
            if J_next.shape != state_dims:
                # same check and message as interp_on_state (:413-415)
                raise ValueError('array `A` should be of shape {:s}, not {:s}'.format(
                    str(state_dims), str(J_next.shape)))
        if report_time:
            print('value iteration...', end='')
        t_k = None
        J_k, J_ref, pol_k, _ = self._sweep_host(J_next, t_k, rel_dp)
        exec_time = (datetime.now() - t_start).total_seconds()
        if report_time:
            print('\rvalue iteration run in {:.2f} s'.format(exec_time))
        if rel_dp:
            J_k = J_k, J_ref
        return J_k, pol_k

    def bellman_recursion(self, t_fin, J_fin, t_ini=0, report_time=True):
        """Bellman backward recursion for finite-horizon problems, from `t_fin`
        down to `t_ini` (must be 0).  Supports time-dependent systems: the instant
        `t_k` is passed first to every callable.

        Returns (J, pol) with a leading time axis.  (reference stodynprog.py:536-591)
        """
        t_start = datetime.now()
        state_dims = tuple(len(g) for g in self.state_grid)
        nb_control = len(self.sys.control)
        print('time-dependent problem: {:s}'.format('no' if self.sys.stationnary else 'yes'))
        assert t_ini == 0  # t_ini > 0 not tested (reference :557)
        J = np.zeros((t_fin - t_ini,) + state_dims)
        pol = np.zeros((t_fin - t_ini,) + state_dims + (nb_control,))
        if report_time:
            print('bellman recursion...', end='')
        J_fin = np.asarray(J_fin)
        if J_fin.shape != state_dims:
            raise ValueError('array `A` should be of shape {:s}, not {:s}'.format(
                str(state_dims), str(J_fin.shape)))
        saved_mode, self.host_results = self.host_results, "all"   # J[k+1] feeds instant k on every rank
        try:
            self._recursion(t_ini, t_fin, J_fin, J, pol)
        finally:
            self.host_results = saved_mode
        exec_time = (datetime.now() - t_start).total_seconds()
        if report_time:
            print('\rvalue iteration run in {:.2f} s'.format(exec_time))
        return J, pol

    def _recursion(self, t_ini, t_fin, J_fin, J, pol):
        # systems whose dynamics and admissible controls ignore the instant (checked, not
        # assumed): one table build, the cost of all instants tabulated up front, the sweeps
        # enqueued back to back (Engine.recursion_fast); anything else: instant by instant
        self.last_recursion = None
        if getattr(self, "recursion_mode", "auto") != "per_instant":
            info = self.engine.recursion_fast(self, t_ini, t_fin, J_fin, J, pol)
            if info is not None:
                self.last_tables = info.pop("tables")
                self.last_recursion = info
                return
        tables = None
        for t_k in range(t_ini, t_fin)[::-1]:
            print('\rtk = {:3d}...'.format(t_k), end='')
            k = t_k - t_ini
            J_next = J_fin if t_k == (t_fin - 1) else J[k + 1]
            # tables depend on t_k: rebuilt each step, device buffers recycled
            tables = self.engine.build_sweep_tables(self, t_k, reuse=tables)
            self.last_tables = tables
            J[k], _, pol[k], _ = self._sweep_host(J_next, t_k, False, tables=tables)

    def eval_policy(self, pol, n_iter, rel_dp=False, J_zero=None,
                    report_time=True, J_ref_full=False):
        """evaluate the policy `pol`: cost of each state after `n_iter` steps
        (the policy-evaluation half of policy iteration).

        With rel_dp the relative DP algorithm is used: after each step the cost
        of the reference state is recorded and subtracted.

        Returns J_pol, or (J_pol, J_ref) if `rel_dp` (J_ref is the last
        reference cost, or the whole history with J_ref_full).
        (reference stodynprog.py:693-775)
        """
        import torch
        t_start = datetime.now()
        state_dims = self._state_grid_shape
        if J_zero is None:
            J_zero = np.zeros(state_dims)
        assert J_zero.shape == state_dims
        ref_ind = self._state_ref_ind
        nb_control = len(self.sys.control)
        assert pol.shape == state_dims + (nb_control,)

        eng = self.engine
        P = eng.build_policy_tables(self, pol)
        n_grid = int(np.prod(state_dims))
        J_a, J_b = eng.J_pair(n_grid)         # symmetric (peer-mapped) buffers with several ranks
        eng.begin_call(n_grid)
        eng.upload_J(J_zero, J_a)
        hist = torch.zeros(max(n_iter, 1), dtype=torch.float64, device=eng.device)
        ref_flat = int(np.ravel_multi_index(ref_ind, state_dims))
        print('\rpolicy evaluation: iter. {:d}/{:d}'.format(max(n_iter - 1, 0), n_iter), end='')
        J_dev = eng.policy_eval(P, J_a, J_b, n_iter, rel_dp, ref_flat, hist)
        outs = eng.to_host(J_dev, hist)
        J_pol = outs[0].reshape(state_dims)
        J_ref = outs[1][:n_iter] if rel_dp else None

        exec_time = (datetime.now() - t_start).total_seconds()
        if report_time:
            print('\rpolicy evaluation run in {:.2f} s     '.format(exec_time))
        if rel_dp:
            if not J_ref_full:
                J_ref = J_ref[-1]
            return J_pol, J_ref
        return J_pol

    def policy_iteration(self, pol_init, n_val, n_pol=1, rel_dp=False):
        """policy iteration: evaluate `pol_init` with `n_val` fixed-policy
        backups, then `n_pol` times (improve with one value iteration, evaluate).

        Returns (J_pol, pol); J_pol is a tuple (J_diff, J_ref) if `rel_dp`.
        (reference stodynprog.py:777-812)
        """
        saved_mode, self.host_results = self.host_results, "all"   # every rank needs pol to evaluate it
        try:
            return self._policy_iteration(pol_init, n_val, n_pol, rel_dp)
        finally:
            self.host_results = saved_mode

    def _policy_iteration(self, pol_init, n_val, n_pol, rel_dp):
        pol = pol_init
        J_pol = self.eval_policy(pol, n_val, rel_dp)
        if rel_dp:
            J_diff, J_ref = J_pol
            print('ref policy cost: {:g}'.format(J_ref))
        for k in range(n_pol):
            print('policy iteration {:d}/{:d}'.format(k + 1, n_pol))
            _, pol = self.value_iteration(J_pol, rel_dp=rel_dp)
            J_pol = self.eval_policy(pol, n_val, rel_dp)
            if rel_dp:
                J_ref = J_pol[1]
                print('ref policy cost: {:g}'.format(J_ref))
        return J_pol, pol

    # ------------------------------------------------------------------
    # new: device-resident value iteration driven by the sup-norm residual
    # ------------------------------------------------------------------
    def solve_value_iteration(self, J_zero=None, max_iter=100, tol=None, rel_dp=False,
                              check_every=1):
        """Repeated Bellman sweeps with J kept on the device; stops after
        `max_iter` sweeps or when max|J_k - J_{k+1}| <= tol (all-reduced over the
        ranks).  Not in the reference (users write this loop by hand,
        doc/example_inventory.py:98-110).  Returns (J, pol, info)."""
        import torch
        eng = self.engine
        state_dims = tuple(len(g) for g in self.state_grid)
        nb_control = len(self.sys.control)
        T = self.sweep_tables(None)
        J0 = np.zeros(state_dims) if J_zero is None else np.asarray(J_zero, dtype=float)
        n_grid = int(np.prod(state_dims))
        J_prev, J_new = eng.J_pair(n_grid)
        eng.begin_call(n_grid)
        root_only = self._root_only()
        is_root = eng.coll.rank == 0
        if root_only:
            if is_root:
                eng.upload_J(J0, J_prev)
            eng.share_J(J_prev)
        else:
            eng.upload_J(J0, J_prev)
        resid = torch.zeros(1, dtype=torch.float64, device=eng.device)
        ref_out = torch.zeros(1, dtype=torch.float64, device=eng.device) if rel_dp else None
        ref_flat = int(np.ravel_multi_index(self._state_ref_ind, state_dims)) if rel_dp else None
        history = []
        n_done = 0
        for k in range(max_iter):
            # (between two sweeps the arrival of the peers' slabs is awaited by the next sweep's
            # first kernel; relative DP and the residual read J right away and wait themselves)
            eng.sweep(T, J_prev, J_new, rel_ref_index=ref_flat, ref_out=ref_out,
                      resid_out=resid if tol is not None else None, defer_wait=k + 1 < max_iter,
                      want_argmin=(tol is not None or k + 1 == max_iter))
            J_prev, J_new = J_new, J_prev
            n_done += 1
            if tol is not None and (k + 1) % check_every == 0:
                r = float(resid.cpu().numpy()[0])
                history.append(r)
                if r <= tol:
                    break
        eng.flush_exchange()
        argmin_full = eng.gather_argmin(T)
        info = {'n_sweeps': n_done, 'residuals': history,
                'J_ref': float(ref_out.cpu().numpy()[0]) if rel_dp else None}
        if root_only and not is_root:
            return None, None, info
        pol_dev = eng.policy_values(T, argmin_full)
        J, pol = eng.to_host(J_prev, pol_dev)
        J = J.reshape(state_dims)
        pol = pol.reshape(state_dims + (nb_control,))
        return J, pol, info

    # ------------------------------------------------------------------
    # new: what a policy does to the system (forward / adjoint application)
    # ------------------------------------------------------------------
    @staticmethod
    def _check_shape(name, A, expect_shape):
        # same wording as interp_on_state (reference :413-415)
        if A.shape != expect_shape:
            raise ValueError('array `{:s}` should be of shape {:s}, not {:s}'.format(
                name, str(expect_shape), str(A.shape)))

    def _check_mu0(self, mu0):
        mu0 = np.array(mu0, dtype=float)      # a copy: the caller's array is never written
        self._check_shape('mu0', mu0, self._state_grid_shape)
        if not np.all(np.isfinite(mu0)):
            raise ValueError('`mu0` must be finite')
        return mu0

    def _forward_operator(self, pol, t_k=None):
        eng = self.engine
        P = eng.build_policy_tables(self, np.asarray(pol, dtype=float), t_k=t_k, deterministic=True)
        return eng.build_forward(P)

    def propagate_distribution(self, pol, mu0, n_steps=None, history=False, report_time=True):
        """distribution of the state after `n_steps` steps under the policy `pol`, starting
        from the distribution `mu0` on the state grid, and the expected stage cost of every
        step.  Not in the reference (which simulates trajectories one point at a time).

        The chain is the one the value function is computed with: the next state of a grid
        point is spread over the corners of its cell with the interpolation weights (the
        exact transpose of eval_policy's backup).  Next states outside the grid box
        extrapolate, which can give negative mass near the boundary.  The operator is
        linear, so `mu0` need not be normalised.

        Stationary systems: `pol` of shape state_dims + (nb_control,), `n_steps` required.
        Time-dependent systems: `pol` of shape (T,) + state_dims + (nb_control,) as returned
        by bellman_recursion; step k applies pol[k] at instant k; `n_steps` defaults to T.

        Returns (mu, expected_cost): mu_n of shape state_dims (or the history mu_0 .. mu_n,
        shape (n_steps+1,) + state_dims, with `history`), and expected_cost[k] =
        sum_x mu_k(x) * sum_w p_w g(x, pol(x), w), k < n_steps.
        """
        import torch
        t_start = datetime.now()
        state_dims = self._state_grid_shape
        nb_control = len(self.sys.control)
        pol = np.asarray(pol)
        if self.sys.stationnary:
            self._check_shape('pol', pol, state_dims + (nb_control,))
            if n_steps is None:
                raise ValueError('n_steps is required for a stationary system')
        else:
            T = pol.shape[0] if pol.ndim == len(state_dims) + 2 else 0
            self._check_shape('pol', pol, (max(T, 1),) + state_dims + (nb_control,))
            if n_steps is None:
                n_steps = T
            if n_steps > T:
                raise ValueError('n_steps = {:d} exceeds the horizon of `pol` ({:d} instants)'.format(
                    int(n_steps), T))
        n_steps = int(n_steps)
        if n_steps < 0:
            raise ValueError('n_steps must be >= 0')
        mu0 = self._check_mu0(mu0)
        eng = self.engine
        n = int(np.prod(state_dims))
        if report_time:
            print('distribution propagation...', end='')
        mu_a = eng.to_device(mu0.reshape(-1))
        mu_b = torch.empty_like(mu_a)
        cost = torch.zeros(max(n_steps, 1), dtype=torch.float64, device=eng.device)
        hist = torch.empty((n_steps + 1) * n, dtype=torch.float64, device=eng.device) if history else None
        if self.sys.stationnary:
            F = self._forward_operator(pol)
            mu_n = eng.forward_steps(F, mu_a, mu_b, n_steps, cost, hist=hist)
        else:
            # the chain changes with the instant: tables and operator rebuilt per step
            mu_n = mu_a
            for k in range(n_steps):
                F = self._forward_operator(pol[k], t_k=k)
                nxt = mu_b if mu_n is mu_a else mu_a
                eng.forward_steps(F, mu_n, nxt, 1, cost[k:k + 1],
                                  hist=hist[k * n:(k + 2) * n] if history else None)
                mu_n = nxt
                del F
        mu, cost_h = eng.to_host(hist if history else mu_n, cost)
        exec_time = (datetime.now() - t_start).total_seconds()
        if report_time:
            print('\rdistribution propagation run in {:.2f} s'.format(exec_time))
        shape = ((n_steps + 1,) if history else ()) + state_dims
        return mu.reshape(shape), cost_h[:n_steps].copy()

    def stationary_distribution(self, pol, mu0=None, tol=1e-12, max_iter=100_000, check_every=50,
                                report_time=True):
        """stationary distribution pi = P^T pi of the chain of the stationary policy `pol`
        (see propagate_distribution), by power iteration from `mu0` (default: uniform 1/N).
        Stops when sum |mu_{k+1} - mu_k| <= tol, checked every `check_every` steps, or after
        `max_iter` steps; a chain that does not converge returns converged=False.  The
        operator is linear, so `mu0` need not be normalised (tol is then relative to its mass).
        Not in the reference.

        Returns (pi, info): pi of shape state_dims, info = {'n_steps', 'converged',
        'residuals' (one per check), 'average_cost' = sum_x pi(x) g_bar(x), 'mass' = sum pi,
        'negative_mass' = sum min(pi, 0)} - negative mass means the grid is too small for the
        policy's next states (they extrapolate out of the grid box).
        """
        t_start = datetime.now()
        if not self.sys.stationnary:
            raise ValueError('stationary_distribution needs a stationary system')
        state_dims = self._state_grid_shape
        pol = np.asarray(pol)
        self._check_shape('pol', pol, state_dims + (len(self.sys.control),))
        n = int(np.prod(state_dims))
        mu0 = np.full(state_dims, 1.0 / n) if mu0 is None else self._check_mu0(mu0)
        if int(max_iter) < 0 or int(check_every) < 1:
            raise ValueError('max_iter must be >= 0 and check_every >= 1')
        if report_time:
            print('stationary distribution...', end='')
        eng = self.engine
        F = self._forward_operator(pol)
        pi_dev, n_done, residuals, converged = eng.stationary(F, mu0, tol, int(max_iter), int(check_every))
        pi, gbar = eng.to_host(pi_dev, F.bufs["gbar"])
        pi = pi.reshape(state_dims)
        info = {'n_steps': n_done, 'converged': converged, 'residuals': residuals,
                'average_cost': float(np.dot(pi.reshape(-1), gbar)),
                'mass': float(pi.sum()), 'negative_mass': float(np.minimum(pi, 0).sum())}
        exec_time = (datetime.now() - t_start).total_seconds()
        if report_time:
            print('\rstationary distribution run in {:.2f} s ({:d} steps)'.format(exec_time, n_done))
        return pi, info

    def _check_start(self, start, n_paths):
        """(flat start indices int32 [n_paths], None) or (None, C-order CDF of the start distribution)"""
        state_dims = self._state_grid_shape
        n = int(np.prod(state_dims))
        if isinstance(start, tuple):
            if len(start) != len(state_dims) or not all(isinstance(i, (int, np.integer)) for i in start) or \
                    not all(0 <= i < m for i, m in zip(start, state_dims)):
                raise ValueError('`start` as a tuple should be a multi-index of the state grid of shape {:s}, '
                                 'not {:s}'.format(str(state_dims), str(start)))
            return np.full(n_paths, np.ravel_multi_index(start, state_dims), dtype=np.int32), None
        start = np.asarray(start)
        if np.issubdtype(start.dtype, np.integer):
            self._check_shape('start', start, (n_paths,))
            if start.size and (start.min() < 0 or start.max() >= n):
                raise ValueError('flat indices in `start` must lie in [0, {:d})'.format(n))
            return start.astype(np.int32), None
        if not np.issubdtype(start.dtype, np.floating):
            raise ValueError('`start` should be a multi-index (tuple), an integer array of flat indices or '
                             'a distribution (float array)')
        self._check_shape('start', start, state_dims)
        if not np.all(np.isfinite(start)) or np.any(start < 0) or not start.sum() > 0:
            raise ValueError('the start distribution must be finite, non-negative and not all zero')
        return None, np.cumsum(start.reshape(-1).astype(float))

    def _chain_tables(self, pol, t_k=None):
        eng = self.engine
        P = eng.build_policy_tables(self, np.asarray(pol, dtype=float), t_k=t_k, deterministic=True)
        return eng.chain_tables(P)

    def sample_paths(self, pol, start, n_steps, n_paths, seed=0, target=None, record=(), report_time=True):
        """sample `n_paths` paths of `n_steps` steps of the chain of the policy `pol` (Monte-Carlo
        trajectories on the GPU, one thread per path).  Not in the reference as such: its
        examples simulate the policy on the host.

        The chain is the one of propagate_distribution, sampled: from state x a perturbation node
        w is drawn with its probability, then the next state's cell corner along every axis k is
        the upper one with probability lambda_k, the interpolation weight; the stage cost
        g(x, pol(x), w) is added to the path's total.  Where a next state lies outside the grid
        box, lambda_k is outside [0, 1] and is clamped to it (a probability cannot be negative):
        the sample projects that next state onto the grid box.  Such transitions are counted
        (info['clamped_share']); with none, the sampled chain is exactly the chain J is computed
        with.  A NaN weight takes the lower corner and is counted in info['nan_transitions'].

        Random numbers are Philox-4x32-10 keyed by `seed`, counter (path, step, call): a path's
        results depend only on (seed, path index, policy), and are bit-identical run to run.

        pol: state_dims + (nb_control,) for a stationary system; (T,) + state_dims + (nb_control,)
            as returned by bellman_recursion for a time-dependent one (step k applies pol[k] at
            instant k, n_steps <= T).
        start: a tuple, the multi-index every path starts from; an integer array of n_paths flat
            C-order indices; or a float array of shape state_dims, non-negative, the (not
            necessarily normalised) distribution the initial states are drawn from.
        target: boolean array of shape state_dims, or None.
        record: steps in [0, n_steps] at which the states are returned.

        Returns (total_cost [n_paths], info) with info = {'hit_step' [n_paths]: first step (0 ..
        n_steps) at which the path is in `target`, -1 if never; 'states' [len(record), n_paths]:
        flat indices of the states at the recorded steps; 'final_state' [n_paths]; 'clamped_share';
        'nan_transitions'; 'n_paths'; 'n_steps'; 'seed'}.
        """
        import torch
        t_start = datetime.now()
        state_dims = self._state_grid_shape
        nb_control = len(self.sys.control)
        pol = np.asarray(pol)
        if self.sys.stationnary:
            self._check_shape('pol', pol, state_dims + (nb_control,))
        else:
            T = pol.shape[0] if pol.ndim == len(state_dims) + 2 else 0
            self._check_shape('pol', pol, (max(T, 1),) + state_dims + (nb_control,))
        n_steps, n_paths, seed = int(n_steps), int(n_paths), int(seed)
        if n_steps < 0:
            raise ValueError('n_steps must be >= 0')
        if not self.sys.stationnary and n_steps > T:
            raise ValueError('n_steps = {:d} exceeds the horizon of `pol` ({:d} instants)'.format(n_steps, T))
        if not 1 <= n_paths < 2 ** 31:
            raise ValueError('n_paths must be in [1, 2**31), not {:d}'.format(n_paths))
        if not 0 <= seed < 2 ** 64:
            raise ValueError('seed must be in [0, 2**64)')
        start_idx, start_cdf = self._check_start(start, n_paths)
        if target is not None:
            target = np.asarray(target)
            self._check_shape('target', target, state_dims)
            if target.dtype != bool:
                raise ValueError('`target` must be a boolean array')
        record = np.asarray(record)
        if record.size and not np.issubdtype(record.dtype, np.integer):
            raise ValueError('`record` must hold integer steps')
        record = record.astype(np.int64).reshape(-1)
        if np.any((record < 0) | (record > n_steps)):
            raise ValueError('`record` steps must lie in [0, n_steps] = [0, {:d}]'.format(n_steps))
        rec_steps, rec_inv = np.unique(record, return_inverse=True)
        if report_time:
            print('path sampling...', end='')
        eng = self.engine
        dev = eng.device
        M = n_paths
        state = eng.to_device(start_idx) if start_idx is not None else \
            torch.empty(M, dtype=torch.int32, device=dev)
        total = torch.empty(M, dtype=torch.float64, device=dev)
        hit = torch.empty(M, dtype=torch.int32, device=dev)
        counters = torch.zeros(2, dtype=torch.int64, device=dev)
        kw = {"start_cdf": eng.to_device(start_cdf) if start_cdf is not None else None,
              "target": eng.to_device(self._target_mask(target)) if target is not None else None,
              "rec_steps": eng.to_device(rec_steps.astype(np.int32)) if rec_steps.size else None,
              "rec_out": torch.empty(rec_steps.size * M, dtype=torch.int32, device=dev) if rec_steps.size else None}
        if self.sys.stationnary:
            C = self._chain_tables(pol)
            eng.chain_sample(C, state, total, hit, n_steps, 0, seed, True, counters, **kw)
        else:
            # the chain changes with the instant: tables rebuilt per step, the paths resume on the
            # device with the global step in the random counter
            for k in range(max(n_steps, 1)):
                C = self._chain_tables(pol[k], t_k=k)
                eng.chain_sample(C, state, total, hit, min(n_steps, 1), k, seed, k == 0, counters, **kw)
                del C
        outs = [total, hit, state, counters] + ([kw["rec_out"]] if rec_steps.size else [])
        host = eng.to_host(*outs)
        total_h, hit_h, final_h, cnt = host[:4]
        states = host[4].reshape(rec_steps.size, M)[rec_inv] if rec_steps.size else np.zeros((0, M), np.int32)
        info = {'hit_step': hit_h, 'states': states, 'final_state': final_h,
                'clamped_share': float(cnt[0]) / (M * n_steps) if n_steps else 0.0,
                'nan_transitions': int(cnt[1]), 'n_paths': M, 'n_steps': n_steps, 'seed': seed}
        exec_time = (datetime.now() - t_start).total_seconds()
        if report_time:
            print('\rpath sampling run in {:.2f} s ({:d} paths x {:d} steps)'.format(exec_time, M, n_steps))
        return total_h, info

    def first_passage(self, pol, target, n_steps=None, clamp=True, history=False, tol=None, check_every=50,
                      report_time=True):
        """first-passage analysis of the chain of the policy `pol` with respect to the set
        `target`, exact and for every start state at once (a backward recursion on the GPU, one
        thread per state).  Not in the reference.

        Let tau be the first step k >= 0 at which the path is in `target` (a start in the target
        gives tau = 0, as sample_paths' hit_step).  Over a horizon of n = n_steps steps this returns,
        for every start state x:
            prob[x]  = P_x(tau <= n), the probability of reaching the target within n steps;
            steps[x] = E_x[min(tau, n)], the expected number of steps before reaching it;
            cost[x]  = the expected stage cost accumulated before tau, within the horizon.
        They are computed backwards from (1_target, 0, 0) at step n: off the target,
        P_k = sum_w p_w I[P_{k+1}](f(x, w)), S_k = 1 + sum_w p_w I[S_{k+1}], C_k = sum_w p_w (g + I[C_{k+1}]),
        with I the multilinear interpolation at the next state; on the target (1, 0, 0).

        clamp=True (default): the interpolation weights are clamped to [0, 1] (NaN: 0), the chain
            sample_paths samples, so that prob is a true probability.  clamp=False: the weights are
            used as they are, the chain J is computed with (eval_policy, propagate_distribution);
            near the boundary its values can leave [0, 1].  With an empty target and clamp=False,
            cost is eval_policy(pol, n) bit for bit.
        pol: state_dims + (nb_control,) for a stationary system (n_steps required); (T,) +
            state_dims + (nb_control,) as returned by bellman_recursion for a time-dependent one
            (step k applies pol[k] at instant k; n_steps defaults to T).
        target: boolean array of shape state_dims.
        history: return every V_k, k = 0 .. n: prob, steps, cost of shape (n+1,) + state_dims,
            entry k the values from step k (prob[n] = 1_target).  For a stationary system prob[k]
            is the probability of reaching the target within n - k steps, so the whole law of
            tau from x is P_x(tau <= j) = prob[n - j][x]; from a start distribution mu0 it is
            <mu0, prob[n - j]>.
        tol (stationary systems only): n_steps becomes a maximum; every `check_every` steps the
            sup-norm change of the last step (over the three outputs) is read back, and the
            recursion stops when it is <= tol.  prob then tends to P_x(tau < inf), and steps and
            cost to E_x[tau] and the expected cost before tau wherever the target is reached
            almost surely.  Where it is not, steps grows without bound (by up to one per step)
            and `converged` stays False.

        Returns (prob, steps, cost, info), info = {'n_steps': the steps done, 'converged': whether
        a tol run met tol, 'residuals': the residual read at each check, 'outside_share': the share
        of the (x, w) table entries of non-target states whose weights were clamped (clamp=True)
        or extrapolate (clamp=False), over all the instants used}.
        """
        return self._backward_analysis('first-passage analysis', self.engine.first_passage, pol, np.asarray(target),
                                       n_steps, clamp, history, tol, check_every, report_time, 1.0)

    def cost_moments(self, pol, n_steps=None, target=None, clamp=True, history=False, tol=None, check_every=50,
                     report_time=True):
        """mean, variance and third central moment of the total stage cost of the policy `pol`,
        exact and for every start state at once (a backward recursion on the GPU, one thread per
        state).  Not in the reference: sample_paths estimates the same from one start at a time.

        Let tau be the first step k >= 0 at which the path is in `target` (tau = inf without a
        target) and G = sum_{k < min(tau, n)} g(x_k, pol(x_k), w_k) the stage cost accumulated
        before tau within the horizon of n = n_steps steps.  This returns, for every start state x:
            mean[x]  = E_x[G]  (eval_policy(pol, n) without a target; first_passage's cost with one);
            var[x]   = Var_x[G];
            third[x] = E_x[(G - mean[x])^3].
        The standard deviation is sqrt(var) and the skewness third / var**1.5.  From a start
        distribution mu0 (normalised to sum 1), with mbar = <mu0, mean> and d = mean - mbar:
            E[G] = mbar,  Var[G] = <mu0, var + d**2>,  E[(G - mbar)^3] = <mu0, third + 3 var d + d**3>.
        They are computed backwards from (0, 0, 0) at step n; at each step, off the target, the mean
        m = sum_w p_w (g + I[M](f(x, w))) first, then, with each corner c of the next state's cell
        centred on m, d_c = g + M(c) - m: V = sum_w p_w I[V(c) + d_c**2],
        K = sum_w p_w I[K(c) + d_c (3 V(c) + d_c**2)] (the laws of total variance and total
        cumulance; I the multilinear interpolation at the next state); on the target (0, 0, 0).
        The centred form keeps the digits that E[G**2] - mean**2 would lose where the mean is large
        against the spread, and with clamp=True var >= 0 holds exactly.

        clamp=True (default): the interpolation weights are clamped to [0, 1] (NaN: 0), the chain
            sample_paths samples.  clamp=False: the weights are used as they are, the chain J is
            computed with.
        pol: state_dims + (nb_control,) for a stationary system (n_steps required); (T,) +
            state_dims + (nb_control,) as returned by bellman_recursion for a time-dependent one
            (step k applies pol[k] at instant k; n_steps defaults to T).  Deterministic systems
            are accepted.
        target: boolean array of shape state_dims, or None (the cost over the whole horizon).
        history: return every step k = 0 .. n: mean, var, third of shape (n+1,) + state_dims.  For
            a stationary system entry k holds the moments of the cost over the last n - k steps,
            so it shows how the spread grows with the horizon.
        tol (stationary systems with a target only): n_steps becomes a maximum; every
            `check_every` steps the sup-norm change of the last step (over the three outputs) is
            read back, and the recursion stops when it is <= tol: the moments of the cost before
            tau, wherever tau is almost surely finite.  Without a target the mean and variance grow
            without bound.

        Returns (mean, var, third, info), info = {'n_steps': the steps done, 'converged': whether a
        tol run met tol, 'residuals': the residual read at each check, 'outside_share': the share of
        the (x, w) table entries of non-target states whose weights were clamped (clamp=True) or
        extrapolate (clamp=False), over all the instants used}.
        """
        if target is not None:
            target = np.asarray(target)
        elif tol is not None:
            raise ValueError('tol needs a target: without one the moments grow without bound')
        return self._backward_analysis('cost moments', self.engine.cost_moments, pol, target, n_steps, clamp,
                                       history, tol, check_every, report_time, 0.0)

    def _backward_analysis(self, what, run, pol, target, n_steps, clamp, history, tol, check_every, report_time,
                           on_target):
        """the driver of first_passage and cost_moments: the argument checks, then n_steps steps of
        the backward recursion `run` (Engine.first_passage or .cost_moments) from the records
        (on_target if the state is in `target` else 0, 0, 0, 0); stationary systems in chunks of
        check_every steps when tol is given, time-dependent ones instant by instant from n-1 to 0.
        target: boolean state_dims array, or None (no target, no mask).  Returns the first three
        values of the records (with `history`, every step, entry k = step k) and info."""
        import torch
        t_start = datetime.now()
        state_dims = self._state_grid_shape
        nb_control = len(self.sys.control)
        pol = np.asarray(pol)
        if self.sys.stationnary:
            self._check_shape('pol', pol, state_dims + (nb_control,))
            if n_steps is None:
                raise ValueError('n_steps is required for a stationary system')
        else:
            T = pol.shape[0] if pol.ndim == len(state_dims) + 2 else 0
            self._check_shape('pol', pol, (max(T, 1),) + state_dims + (nb_control,))
            if n_steps is None:
                n_steps = T
            if n_steps > T:
                raise ValueError('n_steps = {:d} exceeds the horizon of `pol` ({:d} instants)'.format(
                    int(n_steps), T))
            if tol is not None:
                raise ValueError('tol needs a stationary system')
        n_steps = int(n_steps)
        if n_steps < 0:
            raise ValueError('n_steps must be >= 0')
        if int(check_every) < 1:
            raise ValueError('check_every must be >= 1')
        if target is not None:
            self._check_shape('target', target, state_dims)
            if target.dtype != bool:
                raise ValueError('`target` must be a boolean array')
        if report_time:
            print(what + '...', end='')
        eng = self.engine
        n = int(np.prod(state_dims))
        V0 = np.zeros((n, 4))
        if target is not None:
            V0[:, 0] = np.where(target.reshape(-1), on_target, 0.0)
        V_a = eng.to_device(V0.reshape(-1))
        V_b = torch.empty_like(V_a)
        mask = eng.to_device(self._target_mask(target)) if target is not None else None
        counters = torch.zeros(1, dtype=torch.int64, device=eng.device)
        hist = torch.empty((n_steps + 1) * n * 4, dtype=torch.float64, device=eng.device) if history else None
        residuals, converged, done, entries = [], False, 0, 0
        if self.sys.stationnary:
            P = eng.build_policy_tables(self, np.asarray(pol, dtype=float), deterministic=True)
            chunk = n_steps if tol is None else int(check_every)
            resid = torch.zeros(1, dtype=torch.float64, device=eng.device) if tol is not None else None
            while True:
                k = min(chunk, n_steps - done)
                out = run(P, mask, clamp, V_a, V_b, k, counters=counters, resid_out=resid,
                          hist=hist[done * n * 4:(done + k + 1) * n * 4] if history else None)
                if out is V_b:
                    V_a, V_b = V_b, V_a
                done += k
                entries += P.W * n if k else 0
                if tol is not None and k > 0:
                    r = float(resid.cpu().numpy()[0])
                    residuals.append(r)
                    if r <= tol:
                        converged = True
                        break
                if done >= n_steps:
                    break
        else:
            # the chain changes with the instant: tables rebuilt per step, swept from instant n-1 to 0
            for k in range(n_steps - 1, -1, -1):
                P = eng.build_policy_tables(self, np.asarray(pol[k], dtype=float), t_k=k, deterministic=True)
                j = n_steps - 1 - k
                run(P, mask, clamp, V_a, V_b, 1, counters=counters,
                    hist=hist[j * n * 4:(j + 2) * n * 4] if history else None)
                V_a, V_b = V_b, V_a
                done += 1
                entries += P.W * n
                del P
        V, cnt = eng.to_host(hist if history else V_a, counters)
        if history:
            V = V[:(done + 1) * n * 4].reshape(done + 1, n, 4)[::-1]
        shape = ((done + 1,) if history else ()) + state_dims
        V = V.reshape(shape[:-len(state_dims)] + (n, 4))
        a, b, c = (np.ascontiguousarray(V[..., j]).reshape(shape) for j in range(3))
        info = {'n_steps': done, 'converged': converged, 'residuals': residuals,
                'outside_share': float(cnt[0]) / entries if entries else 0.0}
        exec_time = (datetime.now() - t_start).total_seconds()
        if report_time:
            print('\r{:s} run in {:.2f} s ({:d} steps)'.format(what, exec_time, done))
        return a, b, c, info

    @staticmethod
    def _target_mask(target):
        """boolean state_dims array -> 32-bit words, bit y % 32 of word y // 32 = target[y] (C order)"""
        bits = np.packbits(target.reshape(-1), bitorder='little')
        bits = np.concatenate([bits, np.zeros(-bits.size % 4, np.uint8)])
        return bits.view('<i4').astype(np.int32)      # the same bits; torch copies int32

    # ------------------------------------------------------------------
    def print_summary(self):
        """summary of the discretisation (reference stodynprog.py:814-875)"""
        print('SDP solver for system "{}"'.format(self.sys.name))
        grid_size = 'x'.join([str(len(grid)) for grid in self.state_grid])
        print('* state space discretized on a {:s} points grid'.format(grid_size))
        for i, grid in enumerate(self.state_grid):
            if len(grid) > 1:
                print('  - Δ{:s} = {:g}'.format(self.sys.state[i], grid[1] - grid[0]))
            else:
                print('  - {:s} fixed at {:g}'.format(self.sys.state[i], grid[0]))

        if self.sys.stochastic:
            grid_size = 'x'.join([str(len(grid)) for grid in self.perturb_grid])
            print('* perturbation discretized on a {:s} points grid'.format(grid_size))
            for i, grid in enumerate(self.perturb_grid):
                if len(grid) > 1:
                    print('  - Δ{:s} = {:g}'.format(self.sys.perturb[i], grid[1] - grid[0]))
                else:
                    print('  - {:s} fixed at {:g}'.format(self.sys.perturb[i], grid[0]))

        cdim = None
        t_k = None if self.sys.stationnary else 0
        if self.sys.control_box is not None:
            dims = [self.control_grids(x_k, t_k)[1] for x_k in itertools.product(*self.state_grid)]
            cdim = np.array(dims)
        else:
            print('Warning: sys.control_box is still to be defined!')

        print('* control discretization steps:')
        for i in range(len(self.sys.control)):
            print('  - Δ{:s} = {:g}'.format(self.sys.control[i], self.control_steps[i]))
            if cdim is not None and len(cdim):
                if cdim[:, i].min() != cdim[:, i].max():
                    print(('    yields [{:,d} to {:,d}] possible values'
                           ' ({:,.1f} on average)').format(
                        cdim[:, i].min(), cdim[:, i].max(), cdim[:, i].mean()))
                else:
                    print('    yields {:,d} possible values'.format(cdim[0, i]))
        if cdim is not None and len(cdim) and len(self.sys.control) >= 2:
            tot = np.prod(cdim, axis=1)
            print('  control combinations:'
                  ' [{:,d} to {:,d}] possible values ({:,.1f} on average)'.format(
                      tot.min(), tot.max(), tot.mean()))
