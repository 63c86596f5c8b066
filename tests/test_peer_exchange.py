"""The multi-GPU exchange over peer memory, checked on ONE device: N ranks emulated in one process.

Peer pointers are plain device pointers, so the protocol of include/sdp_b200.h (SdpPeers) works
the same when all N ranks live on one GPU.  Every emulated rank owns two J buffers, an int32
argmin buffer, a flag array of N words and an (epoch, done) pair, each a separate allocation
between two guard zones; the four SdpPeers of a rank (J buffer 0 / 1, with and without A[]) are
built as PeerExchange builds them.  Covered: the fused combines (`sdp_sweep_finalize_p2p` on
shards of rows in every layout, `sdp_sweep_finalize_p2p_cols` on shards of columns), the flag
wait folded into the column-table pre-pass (`sdp_sweep_partials_after`) and its non-folding
branches, the fixed-policy backup with relative DP (`sdp_policy_eval_p2p`), `sdp_p2p_broadcast`,
`sdp_p2p_wait`, `sdp_p2p_barrier`, and the argument checks of all of them.  Every rank's buffers
must equal the single-rank result bit for bit, and that result the oracle port.

After every call the harness checks that the guard zones are untouched, that epoch[r] is the
number of publishing calls rank r has made, that flags[q][r] == epoch[r] on every rank q and
that done[r] == 0.

Hang-free discipline (every test here keeps it; a new test must too):
* all emulated ranks are enqueued on ONE stream, in rank order, never on a stream per rank: the
  folded wait spins in every CTA of the pre-pass and could keep a peer's combine from running;
* before an `sdp_p2p_wait`, `sdp_sweep_partials_after` or `sdp_p2p_barrier` of rank r is
  enqueued, the host synchronises and asserts that every flag it will wait on already holds the
  epoch it waits for: a protocol bug fails an assertion instead of spinning;
* the barriers run with the flags of the ranks that come later pre-written by the host, with
  exactly the value those ranks will publish, once in rank order and once in reverse order;
* `p2p_timeout_s` is 10 s for this module (a wait that is wrong anyway traps instead of hanging)
  and 600 s again afterwards.

Tests marked with the "model" backend run the same harness on tests/fake_lib.py (numpy models of
the entry points, which raise on a wait for an unpublished flag) in the CPU suite."""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import ROOT, rel_err
from test_parity import (J_RTOL, _Api, _column_case, _factor_case, _same_bits, _toy, _two_control_system)

gpu = pytest.mark.gpu
BACKENDS = [pytest.param("model"), pytest.param("cuda", marks=gpu)]

GUARD = 0x7ff4dead0000beef        # a NaN bit pattern no kernel writes
GW = 32                            # guard words before and after every allocation
SENT_J = -8.125e300                # destination sentinel: no J of these problems comes near it
SENT_A = -77


@pytest.fixture(scope="module", autouse=True)
def _flag_timeout(product):
    from stodynprog_b200 import _cabi
    lib = _cabi.load_library()
    _cabi.check(lib.sdp_set_option(b"p2p_timeout_s", 10), "sdp_set_option")
    yield
    lib.sdp_set_option(b"p2p_timeout_s", 600)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr())


def _np(t):
    return t.detach().cpu().numpy().copy()


class Ranks(object):
    """N ranks of the peer exchange emulated on the engine's device (see the module docstring)"""

    def __init__(self, eng, N, n_grid):
        import torch
        from stodynprog_b200 import _cabi
        self.eng, self.N, self.n = eng, N, n_grid
        self._alloc = []

        def alloc(words):
            t = torch.full((words + 2 * GW,), GUARD, dtype=torch.int64, device=eng.device)
            self._alloc.append(t)
            return t[GW:GW + words]
        self.J = [[alloc(n_grid).view(torch.float64) for _ in range(2)] for _ in range(N)]
        self.A = [alloc((n_grid + 1) // 2).view(torch.int32)[:n_grid] for _ in range(N)]
        self.flags = [alloc(N) for _ in range(N)]
        self.ed = [alloc(2) for _ in range(N)]          # [epoch, done (low 32 bits)]
        for t in self.flags + self.ed:
            t.zero_()
        self.calls = [0] * N
        self.peers = []
        for r in range(N):
            per = {}
            for k in range(2):
                for with_a in (True, False):
                    P = _cabi.SdpPeers()
                    P.world, P.rank = N, r
                    for q in range(N):
                        P.J[q] = self.J[q][k].data_ptr()
                        P.flags[q] = self.flags[q].data_ptr()
                        P.A[q] = self.A[q].data_ptr() if with_a else None
                    P.epoch = self.ed[r].data_ptr()
                    P.done = self.ed[r].data_ptr() + 8
                    per[k, with_a] = P
            self.peers.append(per)

    def sync(self):
        if self.eng._cuda:
            import torch
            torch.cuda.synchronize(self.eng.device)

    def fill(self, k):
        """destination sentinels before a sweep: J buffer k and the argmin buffer of every rank"""
        for r in range(self.N):
            self.J[r][k].fill_(SENT_J)
            self.A[r].fill_(SENT_A)

    def check(self, flags=True):
        import torch
        self.sync()
        g = torch.cat([torch.cat([t[:GW], t[-GW:]]) for t in self._alloc]).cpu().numpy()
        assert np.all(g == GUARD), "a guard zone was written"
        E = np.stack([_np(e) for e in self.ed])
        assert [int(e) for e in E[:, 0]] == self.calls, (E[:, 0], self.calls)
        assert np.all(E[:, 1] == 0), E[:, 1]
        if flags:
            F = np.stack([_np(f) for f in self.flags])          # F[q][r]: rank r's flag on rank q
            assert np.all(F == E[:, 0][None, :]), F

    def published(self, r):
        self.calls[r] += 1
        self.check()

    def ready(self, r, e=None, skip_own=False):
        """host side, before a wait of rank r is enqueued: every flag it waits on holds epoch e
        (skip_own: but its own, which the barrier kernel writes before it waits)"""
        self.sync()
        e = self.calls[r] if e is None else e
        f = _np(self.flags[r])
        if skip_own:
            f[r] = e
        assert np.all(f >= e), "rank %d would wait for epoch %d on flags %s" % (r, e, list(f))

    def wait(self, r):
        from stodynprog_b200 import _cabi
        self.ready(r)
        _cabi.check(self.eng.lib.sdp_p2p_wait(ctypes.byref(self.peers[r][0, True]), self.eng.stream),
                    "sdp_p2p_wait")
        self.check()

    def wait_all(self):
        for r in range(self.N):
            self.wait(r)

    def load(self, k, J):
        """J (host) into buffer k of every rank"""
        Jd = self.eng.to_device(np.ascontiguousarray(J, dtype=np.float64).reshape(-1))
        for r in range(self.N):
            self.J[r][k].copy_(Jd)
        self.sync()


# ---------------------------------------------------------------------------
# helpers: shards, single-rank reference, one exchanged sweep
# ---------------------------------------------------------------------------
LAYOUTS = {"A": ("control_minor", "auto", "off", "off"), "B": ("state_minor", "auto", "off", "off"),
           "AF": ("control_minor", "auto", "on", "off"), "BF": ("state_minor", "auto", "on", "off"),
           "CF": ("state_minor", "auto", "on", "on")}
LAYOUT_NAMES = {"A": "control_minor", "B": "state_minor", "AF": "control_minor_factored",
                "BF": "state_minor_factored", "CF": "column_factored"}


def _case(api, which):
    """the problems of these tests: the factored and column cases of test_parity, and grids with
    enough columns for 8 shards of columns"""
    import workloads as wl
    if which.startswith("ar1_70x70_w"):
        # 70 rows (3 tiles per column, the last with padding), 70 columns: shards wider than 32
        return wl.storage_ar1(api, n_E=70, n_P=70, n_w=int(which[11:]), steps=(0.5, 0.1)).solver
    if which == "curtail_9":
        sv = _two_control_system(api)                 # two controls, 9 columns
        sv.discretize_state(0, 10., 35, -4, 4, 9)
        return sv
    if which == "config5":
        return wl.storage_ar1_large(api).solver
    if which.startswith("ar1_w") or which in ("searev_col",):
        return _column_case(api, "searev" if which == "searev_col" else which)
    return _factor_case(api, which)


def _maker(product, backend, layout, which, pairs="off"):
    def make():
        sv = _case(_Api(product, backend, *LAYOUTS[layout]), which)
        if layout == "CF":
            sv.column_pairs = pairs
        return sv
    return make


def _shards(make, cuts, axis):
    """(solver, tables) of every rank: states [cuts[r], cuts[r+1]) (rows) or the columns
    [cuts[r], cuts[r+1]) of every row (columns), through the one-shard hooks of the table build"""
    out = []
    for r in range(len(cuts) - 1):
        sv = make()
        c0, c1 = cuts[r], cuts[r + 1]
        setattr(sv, "_slab_override" if axis == "rows" else "_col_override", (c0, c1))
        T = sv.sweep_tables()
        if axis == "rows":
            assert (T.state_begin, T.n_states) == (c0, c1 - c0)
        else:
            # (under the override the tables name their own cut, not the global one)
            assert T.column and T.col_bounds == [c0, c1] and T.n_cols == c1 - c0
        out.append((sv, T))
    return out


def _full_sweeps(sv, J0, n_sweeps=1, inject=False):
    """n single-rank sweeps of the whole grid through the raw ABI (sdp_sweep_partials +
    sdp_sweep_finalize, device-resident): [(J, argmin)] in grid order; inject: NaN / inf into the
    input of the fourth sweep, as test_column_prune._check_sweeps does"""
    import torch
    from stodynprog_b200 import _cabi
    eng, T = sv.engine, sv.sweep_tables()
    n = int(np.prod(sv._state_grid_shape))
    Jp = eng.to_device(np.ascontiguousarray(J0, dtype=np.float64).reshape(-1))
    out = []
    for s in range(n_sweeps):
        Jo = torch.empty_like(Jp)
        A = torch.empty(n, dtype=torch.int32, device=eng.device)
        _cabi.check(eng.lib.sdp_sweep_partials(ctypes.byref(T.grid), ctypes.byref(T.c_tables), _ptr(Jp),
                                               _ptr(T.part_val), _ptr(T.part_idx), eng.stream), "sdp_sweep_partials")
        _cabi.check(eng.lib.sdp_sweep_finalize(ctypes.byref(T.c_tables), _ptr(T.part_val), _ptr(T.part_idx),
                                               _ptr(Jo), _ptr(A), eng.stream), "sdp_sweep_finalize")
        out.append((_np(Jo), _np(A)))
        Jp = Jo
        if inject and s == 2:
            Jp = eng.to_device(_injected(out[-1][0]))
    return out


def _injected(J):
    J = J.copy()
    J[::7] = np.nan
    J[3::11] = np.inf
    return J


def _exchange(em, shards, k_prev, k_new, with_a, glob_cols=None, cuts=None, after=False, tables=None):
    """one sweep of every rank, in rank order on the one stream: partial minima from the rank's own
    copy of J[k_prev] - after=True: sdp_sweep_partials_after on the peers of the previous sweep, once
    the host has seen their flags - then the fused combine into J[k_new] of every rank.  glob_cols:
    shards of columns (sdp_sweep_finalize_p2p_cols at col_begin = cuts[r]).  Returns the launches of
    every rank's partials call."""
    from stodynprog_b200 import _cabi
    eng = em.eng
    lib = eng.lib
    launches = []
    for r, (sv, T) in enumerate(shards):
        c = T.c_tables if tables is None else tables[r]
        args = (ctypes.byref(T.grid), ctypes.byref(c), _ptr(em.J[r][k_prev]), _ptr(T.part_val), _ptr(T.part_idx))
        n0 = lib.sdp_launch_count()
        if after:
            em.ready(r)
            _cabi.check(lib.sdp_sweep_partials_after(*(args + (ctypes.byref(em.peers[r][k_prev, True]),
                                                                eng.stream))), "sdp_sweep_partials_after")
        else:
            _cabi.check(lib.sdp_sweep_partials(*(args + (eng.stream,))), "sdp_sweep_partials")
        launches.append(lib.sdp_launch_count() - n0)
        P = ctypes.byref(em.peers[r][k_new, with_a])
        if glob_cols is not None:
            rc = lib.sdp_sweep_finalize_p2p_cols(ctypes.byref(c), _ptr(T.part_val), _ptr(T.part_idx), _ptr(T.argmin),
                                                 P, glob_cols, cuts[r], eng.stream)
        else:
            rc = lib.sdp_sweep_finalize_p2p(ctypes.byref(c), _ptr(T.part_val), _ptr(T.part_idx), _ptr(T.argmin),
                                            P, T.state_begin, eng.stream)
        _cabi.check(rc, "sdp_sweep_finalize_p2p")
        em.published(r)
    return launches


def _check_ranks(em, shards, k_new, with_a, J_want, A_want, glob_cols=None, cuts=None, what=""):
    """every rank's J[k_new] and A[] against the single-rank result, every shard's local argmin
    against its slice of it"""
    em.sync()
    for r in range(em.N):
        J = _np(em.J[r][k_new])
        assert _same_bits(J, J_want), (what, "J of rank", r, int((J == SENT_J).sum()))
        A = _np(em.A[r])
        if with_a:
            assert np.array_equal(A, A_want), (what, "A[] of rank", r)
        else:
            assert np.all(A == SENT_A), (what, "A[] written with A NULL", r)
    for r, (sv, T) in enumerate(shards):
        a = _np(T.argmin)[:T.n_states]
        if glob_cols is None:
            want = A_want[T.state_begin:T.state_begin + T.n_states]
        else:
            want = A_want.reshape(-1, glob_cols)[:, cuts[r]:cuts[r + 1]].reshape(-1)
        assert np.array_equal(a, want), (what, "local argmin of rank", r)


def _row_cuts(T_full, N, n_cols, column):
    from stodynprog_b200.engine import partition_by_weight, row_aligned
    U = T_full.host_full.U.astype(np.int64)
    cuts = [int(b) for b in partition_by_weight(U + 1, N)]
    return row_aligned(cuts, n_cols) if column else cuts


def _col_cuts(T_full, N, n_rows, n_cols):
    from stodynprog_b200.engine import partition_by_weight
    col_w = (T_full.host_full.U.astype(np.int64) + 1).reshape(n_rows, n_cols).sum(axis=0)
    cuts = [int(b) for b in partition_by_weight(col_w, N)]
    # (at least one column per shard: a balanced cut of a few uneven columns can leave one empty,
    # which the table build refuses for a shard of columns)
    for i in range(1, N):
        cuts[i] = max(cuts[i], cuts[i - 1] + 1)
    for i in range(N - 1, 0, -1):
        cuts[i] = min(cuts[i], cuts[i + 1] - 1)
    return cuts


def _versus_port(make_port, sv, J0, J_raw):
    """the single-rank full-grid result against the oracle port: policies exact, J <= 1e-10"""
    J, pol = sv.value_iteration(J0, report_time=False)
    assert _same_bits(J.reshape(-1), J_raw)
    with np.errstate(invalid="ignore"):
        Jo, polo = make_port().value_iteration(J0)[:2]
    assert np.array_equal(pol, polo)
    assert rel_err(J, Jo) <= J_RTOL


# ---------------------------------------------------------------------------
# 1. sweeps, shards of rows, every layout
# ---------------------------------------------------------------------------
ROW_CASES = [("A", "storage_ar1"), ("A", "searev"), ("B", "storage_ar1"), ("B", "searev"), ("AF", "uw"),
             ("AF", "storage_ar1"), ("BF", "wu"), ("BF", "storage_ar1"), ("CF", "ar1_w9"), ("CF", "ar1_w3"),
             ("CF", "searev_col")]


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("layout,which", ROW_CASES, ids=["%s-%s" % c for c in ROW_CASES])
def test_row_shards_every_layout(product, port, backend, layout, which, monkeypatch):
    """N = 1, 2, 3, 8 shards of rows: each rank sweeps its own copy of J, the fused combine stores
    into every rank's J and A[]; all equal the single-rank sweep of the whole grid, which equals
    the port"""
    from stodynprog_b200.engine import Engine
    monkeypatch.setattr(Engine, "COLUMN_BANDS", "1")
    make = _maker(product, backend, layout, which)
    full = make()
    T_full = full.sweep_tables()
    assert T_full.layout_name == LAYOUT_NAMES[layout]
    shape = full._state_grid_shape
    n_grid, n_cols = int(np.prod(shape)), int(np.prod(shape[1:]))
    J0 = np.random.default_rng(17).standard_normal(shape)
    (J_want, A_want), = _full_sweeps(full, J0)
    _versus_port(lambda: _case(port, which), full, J0, J_want)
    partial_tile = False
    for N in (1, 2, 3, 8):
        cuts = _row_cuts(T_full, N, n_cols, layout == "CF")
        assert all(b > a for a, b in zip(cuts[:-1], cuts[1:])), cuts
        partial_tile |= any(b % 32 for b in cuts[1:-1])
        shards = _shards(make, cuts, "rows")
        assert all(T.layout_name == LAYOUT_NAMES[layout] for _, T in shards)
        em = Ranks(full.engine, N, n_grid)
        em.load(0, J0)
        em.fill(1)
        _exchange(em, shards, 0, 1, True)
        em.wait_all()
        _check_ranks(em, shards, 1, True, J_want, A_want, what=(layout, which, N))
    assert partial_tile                 # (a cut inside a tile of 32 states: the last tile of a shard is partial)


# ---------------------------------------------------------------------------
# 2. sweeps, shards of columns
# ---------------------------------------------------------------------------
COL_GRIDS = ["ar1_70x70_w3", "ar1_70x70_w9", "searev_col", "curtail_9"]
COL_VARIANTS = [  # (name, col_prune, col_groups, pdl, column_pairs, A[] set)
    ("no_prune", 0, 0, 1, "off", True), ("prune", 1, 0, 1, "off", False), ("groups", 1, 1, 1, "off", True),
    ("groups_no_pdl", 1, 1, 0, "off", False), ("pairs", 1, 1, 1, "on", True)]


def _set_options(lib, prune, groups, pdl):
    """the launch options of a variant; col_threads at its default (0: 640 threads when pruning),
    which group skipping needs, whatever an earlier test left behind"""
    from stodynprog_b200 import _cabi
    for name, v in ((b"col_prune", prune), (b"col_groups", groups), (b"pdl", pdl), (b"col_threads", 0)):
        _cabi.check(lib.sdp_set_option(name, v), "sdp_set_option")


def _restore_options(lib):
    _set_options(lib, 1, 1, 1)
    lib.sdp_set_option(b"dbg_exchange", 0)


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("which", COL_GRIDS)
def test_column_shards(product, port, backend, which, monkeypatch):
    """N = 2, 3, 5, 8 shards of whole columns (sdp_sweep_finalize_p2p_cols, glob_cols and col_begin
    passed explicitly): pruning off / on / with groups, two rows per lane, programmatic dependent
    launch off, A[] NULL and set - every rank's buffers bit-identical to the single-rank sweep"""
    from stodynprog_b200 import _cabi
    from stodynprog_b200.engine import Engine
    if backend == "model" and which.startswith("ar1_70x70"):
        pytest.skip("4 900 states take minutes in the numpy model; covered on the GPU")
    monkeypatch.setattr(Engine, "COLUMN_BANDS", "1")
    full = _maker(product, backend, "CF", which)()
    T_full = full.sweep_tables()
    shape = full._state_grid_shape
    n_grid, n_rows = int(np.prod(shape)), shape[0]
    n_cols = n_grid // n_rows
    J0 = np.random.default_rng(23).standard_normal(shape)
    (J_want, A_want), = _full_sweeps(full, J0)
    _versus_port(lambda: _case(port, which), full, J0, J_want)
    cuda = backend == "cuda"
    lib = full.engine.lib
    wide = False
    try:
        for N in (2, 3, 5, 8):
            cuts = _col_cuts(T_full, N, n_rows, n_cols)
            assert all(b > a for a, b in zip(cuts[:-1], cuts[1:])), cuts
            wide |= max(np.diff(cuts)) > 32
            em = Ranks(full.engine, N, n_grid)
            em.load(0, J0)
            by_pairs = {}
            for name, prune, groups, pdl, pairs, with_a in COL_VARIANTS:
                if not cuda and name not in ("no_prune", "pairs"):
                    continue            # (launch options of the library; the model has none)
                if pairs not in by_pairs:
                    by_pairs[pairs] = _shards(_maker(product, backend, "CF", which, pairs), cuts, "columns")
                shards = by_pairs[pairs]
                assert all(T.pairs == (pairs == "on") for _, T in shards)
                if cuda:
                    _set_options(lib, prune, groups, pdl)
                em.fill(1)
                _exchange(em, shards, 0, 1, with_a, glob_cols=n_cols, cuts=cuts)
                if cuda and groups and pairs == "off":
                    assert "groups" in _cabi.last_kernel(), _cabi.last_kernel()
                em.wait_all()
                _check_ranks(em, shards, 1, with_a, J_want, A_want, n_cols, cuts, what=(which, N, name))
    finally:
        if cuda:
            _restore_options(lib)
    assert wide or which not in ("ar1_70x70_w3", "ar1_70x70_w9")


# ---------------------------------------------------------------------------
# 3. device-resident chains: the flag wait folded into the next sweep's first kernel
# ---------------------------------------------------------------------------
CHAINS = [("rows_CF_folded", "CF", "ar1_w3", "rows"), ("cols_CF_folded", "CF", "ar1_70x70_w3", "columns"),
          ("rows_BF_separate_wait", "BF", "storage_ar1", "rows"), ("rows_CF_table_ready", "CF", "ar1_w3", "rows")]


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("name,layout,which,axis", CHAINS, ids=[c[0] for c in CHAINS])
def test_device_resident_chains(product, backend, name, layout, which, axis, monkeypatch):
    """5 chained sweeps at N = 2, 3, 8: sweep s + 1 starts with sdp_sweep_partials_after on the
    peers of sweep s (no separate wait), NaN / inf injected into J at sweep 2; every rank's buffer
    after every sweep equals the single-rank device sweeps.  Layout CF folds the wait into the
    pre-pass (no extra launch); layout BF, and CF with col_table_ready = 1 (the caller ran the
    pre-pass), launch a separate wait"""
    from stodynprog_b200 import _cabi
    from stodynprog_b200.engine import Engine
    if backend == "model" and which.startswith("ar1_70x70"):
        pytest.skip("4 900 states take minutes in the numpy model; covered on the GPU")
    monkeypatch.setattr(Engine, "COLUMN_BANDS", "1")
    make = _maker(product, backend, layout, which)
    full = make()
    T_full = full.sweep_tables()
    shape = full._state_grid_shape
    n_grid, n_rows = int(np.prod(shape)), shape[0]
    n_cols = n_grid // n_rows
    J0 = np.random.default_rng(29).standard_normal(shape)
    want = _full_sweeps(full, J0, 5, inject=True)
    eng = full.engine
    ready = name.endswith("table_ready")
    for N in (2, 3, 8):
        if axis == "rows":
            cuts, glob = _row_cuts(T_full, N, n_cols, layout == "CF"), None
        else:
            cuts, glob = _col_cuts(T_full, N, n_rows, n_cols), n_cols
        shards = _shards(make, cuts, axis)
        tables = None
        if ready:
            tables = []
            for _, T in shards:
                c = _cabi.SdpTables.from_buffer_copy(T.c_tables)
                c.col_table_ready = 1
                tables.append(c)
        em = Ranks(eng, N, n_grid)
        em.load(0, J0)
        first = None
        for s in range(5):
            k_prev, k_new = s % 2, 1 - s % 2
            em.fill(k_new)
            if ready:
                for r, (sv, T) in enumerate(shards):
                    if s:
                        em.ready(r)      # (the pre-pass reads the peers' slabs of the previous sweep)
                    _cabi.check(eng.lib.sdp_column_table(ctypes.byref(T.grid), ctypes.byref(tables[r]),
                                                         _ptr(em.J[r][k_prev]), eng.stream), "sdp_column_table")
            launches = _exchange(em, shards, k_prev, k_new, True, glob, cuts, after=s > 0, tables=tables)
            if s == 0:
                first = launches
            elif backend == "cuda":
                extra = 0 if (layout == "CF" and not ready) else 1
                assert launches == [n + extra for n in first], (name, launches, first)
            _check_ranks(em, shards, k_new, True, want[s][0], want[s][1], glob, cuts, what=(name, N, s))
            if s == 2:
                J_inj = _injected(want[s][0])
                for r in range(N):
                    em.J[r][k_new].copy_(eng.to_device(J_inj))
        em.wait_all()


# ---------------------------------------------------------------------------
# 4. config #5 (the bench grid) by columns: the pre-pass at 16, 8 and 4 rows per CTA
# ---------------------------------------------------------------------------
def _prepass_rows(n_cols, rows, sms=148):
    """rows per CTA of the column-table pre-pass (launch_column_table): 16, fewer when the shard's
    columns leave SMs idle"""
    TR, col_blocks = 16, (n_cols + 31) // 32
    while TR > 4 and col_blocks * ((rows + TR - 1) // TR) < sms * 6:
        TR >>= 1
    return TR


@gpu
def test_config5_column_shards(product, port, monkeypatch):
    """config #5 (2000 x 500, W = 9) cut into 2, 4 and 8 shards of columns, which run the pre-pass
    at 16, 8 and 4 rows per CTA: two chained sweeps bit-identical to the single-rank sweeps; the
    column tables and bounds the folded-wait pre-pass of the second sweep left behind, read back
    against numpy; 300 seeded states of the first sweep against the port"""
    from test_device_kernels import _ref_bound, _ref_column_tables, _pvals, _read_tables
    from stodynprog_b200.engine import Engine
    monkeypatch.setattr(Engine, "COLUMN_BANDS", "1")
    make = _maker(product, "cuda", "CF", "config5")
    full = make()
    T_full = full.sweep_tables()
    shape = full._state_grid_shape
    n_grid, n_rows = int(np.prod(shape)), shape[0]
    n_cols = n_grid // n_rows
    J0 = np.random.default_rng(11).standard_normal(shape)
    want = _full_sweeps(full, J0, 2)
    ora = _case(port, "config5")
    picks = np.random.default_rng(12).choice(n_grid, size=300, replace=False)
    Ji = ora.interp_on_state(J0)
    want_J = np.empty(300)
    for n, flat in enumerate(picks):
        idx = np.unravel_index(flat, shape)
        want_J[n] = ora.value_at_state(tuple(g[i] for g, i in zip(ora.state_grid, idx)), Ji)[0]
    assert rel_err(want[0][0][picks], want_J) <= J_RTOL
    all_cuts = dict((N, _col_cuts(T_full, N, n_rows, n_cols)) for N in (2, 4, 8))
    del T_full
    reached = {}
    for N, cuts in all_cuts.items():
        shards = _shards(make, cuts, "columns")
        reached[N] = sorted({_prepass_rows(T.n_cols, n_rows) for _, T in shards})
        em = Ranks(full.engine, N, n_grid)
        em.load(0, J0)
        for s in range(2):
            em.fill(1 - s)
            _exchange(em, shards, s, 1 - s, s == 1, n_cols, cuts, after=s == 1)
            _check_ranks(em, shards, 1 - s, s == 1, want[s][0], want[s][1], n_cols, cuts,
                         what=("config5", N, s))
        J1 = want[0][0].reshape(shape)
        for r, (sv, T) in enumerate(shards):
            R = _ref_column_tables(sv, T, J1)
            got = _read_tables(sv, T, _np(T.col_table))
            assert _same_bits(got, R), ("column tables", N, r)
            b = _np(T.col_bound).reshape(-1)[:T.n_cols * n_rows * 2].reshape(T.n_cols, n_rows, 2)
            wb = _ref_bound(R, _pvals(T))
            assert _same_bits(b, wb), ("column bounds", N, r)
        em.wait_all()
        del shards, em
    print("config #5 pre-pass rows per CTA by shard count:", reached)
    assert reached[2] == [16] and reached[4] == [8] and reached[8] == [4], reached


# ---------------------------------------------------------------------------
# 5. empty shards
# ---------------------------------------------------------------------------
EMPTY_CUT = [0, 0, 2, 3, 3, 7, 8, 10, 10]        # ranks 0, 3 and 7 hold no state


def _empty_tables(T_like):
    from stodynprog_b200 import _cabi
    c = _cabi.SdpTables()
    c.W, c.expect, c.layout, c.n_states = T_like.W, T_like.expect, T_like.c_tables.layout, 0
    return c


@pytest.mark.parametrize("backend", BACKENDS)
def test_empty_shards(product, port, backend):
    """the 10 states of the inventory problem (config #1) cut 8 ways with three empty ranks: the
    empty ranks publish (one CTA, nothing stored), the others' sweep and policy backups are those
    of the single rank"""
    import torch
    import workloads as wl
    from stodynprog_b200 import _cabi
    api = _Api(product, backend)
    make = lambda: wl.inventory(api).solver      # noqa: E731
    full = make()
    T_full = full.sweep_tables()
    eng = full.engine
    n_grid = 10
    J0 = np.random.default_rng(3).standard_normal(n_grid)
    (J_want, A_want), = _full_sweeps(full, J0)
    _versus_port(lambda: wl.inventory(port).solver, full, J0, J_want)
    N = len(EMPTY_CUT) - 1
    shards = []
    for r in range(N):
        a, b = EMPTY_CUT[r], EMPTY_CUT[r + 1]
        if b > a:
            sv = make()
            sv._slab_override = (a, b)
            shards.append((sv, sv.sweep_tables()))
        else:
            shards.append((None, None))
    em = Ranks(eng, N, n_grid)
    em.load(0, J0)
    em.fill(1)
    loc_A = torch.full((4,), SENT_A, dtype=torch.int32, device=eng.device)
    for r, (sv, T) in enumerate(shards):
        P = ctypes.byref(em.peers[r][1, True])
        if T is None:
            c = _empty_tables(T_full)
            rc = eng.lib.sdp_sweep_finalize_p2p(ctypes.byref(c), None, None, _ptr(loc_A), P, EMPTY_CUT[r], eng.stream)
        else:
            _cabi.check(eng.lib.sdp_sweep_partials(ctypes.byref(T.grid), ctypes.byref(T.c_tables), _ptr(em.J[r][0]),
                                                   _ptr(T.part_val), _ptr(T.part_idx), eng.stream), "sdp_sweep_partials")
            rc = eng.lib.sdp_sweep_finalize_p2p(ctypes.byref(T.c_tables), _ptr(T.part_val), _ptr(T.part_idx),
                                                _ptr(T.argmin), P, T.state_begin, eng.stream)
        _cabi.check(rc, "sdp_sweep_finalize_p2p")
        em.published(r)
    em.wait_all()
    _check_ranks(em, [s for s in shards if s[1] is not None], 1, True, J_want, A_want, what="inventory")
    assert np.all(_np(loc_A) == SENT_A)
    # the policy path on the same cut
    pol = full.value_iteration(J0, report_time=False)[1]
    _policy_exchange(full, pol, EMPTY_CUT, rel=True, n_iter=6)


# ---------------------------------------------------------------------------
# 6. sdp_policy_eval_p2p
# ---------------------------------------------------------------------------
def _policy_exchange(sv, pol, cuts, rel, n_iter, J_start=None):
    """n_iter fixed-policy backups of every rank's slab of the whole-grid [w][n] planes, fused with
    the exchange (relative DP from each rank's copy of the reference state's entries), against
    sdp_policy_eval on the whole grid, bit for bit; returns (J, J_ref history)"""
    import torch
    from stodynprog_b200 import _cabi
    eng = sv.engine
    shape = sv._state_grid_shape
    d, n = len(shape), int(np.prod(shape))
    P = eng.build_policy_tables(sv, pol)
    W, gpw = P.W, P.g_per_w
    cell = _np(P.cell)[:W * n].reshape(W, n)
    lam = _np(P.lam)[:d * W * n].reshape(d, W, n)
    g = _np(P.g)[:(W if gpw else 1) * n].reshape(-1, n)
    ref = int(np.ravel_multi_index(sv._state_ref_ind, shape))
    J_start = np.zeros(n) if J_start is None else np.ascontiguousarray(J_start, dtype=np.float64).reshape(-1)
    # whole grid, one rank
    Ja, Jb = eng.to_device(J_start.copy()), torch.empty(n, dtype=torch.float64, device=eng.device)
    hist = torch.zeros(n_iter, dtype=torch.float64, device=eng.device)
    _cabi.check(eng.lib.sdp_policy_eval(ctypes.byref(P.grid), W, gpw, _ptr(P.p), _ptr(P.cell), _ptr(P.lam),
                                        P.lam_plane, _ptr(P.g), n, 0, n, _ptr(Ja), _ptr(Jb), n_iter, int(rel), ref,
                                        _ptr(hist) if rel else None, eng.stream), "sdp_policy_eval")
    J_want, h_want = _np(Ja if n_iter % 2 == 0 else Jb), _np(hist)
    # every rank's slab of the planes, sliced on the host; the reference state's entries as
    # build_policy_tables keeps them with several ranks: cell [W], lam [d][W], g [W] or [1]
    N = len(cuts) - 1
    ranks = []
    for r in range(N):
        a, b = cuts[r], cuts[r + 1]
        dev = lambda x: eng.to_device(np.ascontiguousarray(x))      # noqa: E731
        ranks.append(dict(a=a, n=b - a, cell=dev(cell[:, a:b]), lam=dev(lam[:, :, a:b]), g=dev(g[:, a:b]),
                          rc=dev(cell[:, ref]), rl=dev(lam[:, :, ref]), rg=dev(g[:, ref]),
                          hist=torch.full((n_iter,), SENT_J, dtype=torch.float64, device=eng.device)))
    em = Ranks(eng, N, n)
    em.load(0, J_start)
    null = ctypes.c_void_p(0)
    for it in range(n_iter):
        k_in, k_out = it % 2, 1 - it % 2
        em.fill(k_out)
        for r, x in enumerate(ranks):
            empty = x["n"] == 0
            rc = eng.lib.sdp_policy_eval_p2p(
                ctypes.byref(P.grid), W, gpw, _ptr(P.p), null if empty else _ptr(x["cell"]),
                null if empty else _ptr(x["lam"]), W * x["n"], null if empty else _ptr(x["g"]), x["n"], x["a"], n,
                _ptr(em.J[r][k_in]), ctypes.byref(em.peers[r][k_out, False]),
                _ptr(x["rc"]) if rel else null, _ptr(x["rl"]) if rel else null, _ptr(x["rg"]) if rel else null,
                ctypes.c_void_p(x["hist"].data_ptr() + 8 * it) if rel else null, eng.stream)
            _cabi.check(rc, "sdp_policy_eval_p2p")
            em.published(r)
        em.wait_all()
    em.sync()
    for r, x in enumerate(ranks):
        assert _same_bits(_np(em.J[r][n_iter % 2]), J_want), ("policy J of rank", r, cuts, rel)
        if rel:
            assert _same_bits(_np(x["hist"]), h_want), ("J_ref_out of rank", r)
    return J_want, h_want


POLICY_CASES = [(d, kind) for d in (1, 2, 3, 4) for kind in ("plain", "w")] + [(2, "storage_ar1")]


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("d,kind", POLICY_CASES, ids=["%dd-%s" % c for c in POLICY_CASES])
def test_policy_eval_exchange(product, port, backend, d, kind):
    """6 fused policy backups with and without relative DP over 2, 3 and 5 ranks: every rank's J
    equals sdp_policy_eval on the whole grid bit for bit, J_ref_out its J_ref_hist entry, and the
    result the port's eval_policy"""
    import workloads as wl
    api = _Api(product, backend)
    if kind == "storage_ar1":
        sv, so = (wl.storage_ar1(a, n_E=9, n_P=11, steps=(0.01, 0.1)).solver for a in (api, port))
    else:
        sv, so = _toy(api, d, kind), _toy(port, d, kind)
    shape = sv._state_grid_shape
    n = int(np.prod(shape))
    J0 = np.random.default_rng(d).standard_normal(shape)
    pol = sv.value_iteration(J0, report_time=False)[1]
    J_start = np.random.default_rng(40 + d).standard_normal(shape)
    for N in (2, 3, 5):
        cuts = [n * r // N for r in range(N + 1)]
        for rel in (False, True):
            J, h = _policy_exchange(sv, pol, cuts, rel, 6, J_start)
            if N == 2:
                out = so.eval_policy(pol, 6, rel_dp=rel, J_zero=J_start.copy())
                if rel:
                    Jo, refo = out
                    assert abs(h[-1] - refo) <= J_RTOL * abs(refo)
                    assert np.max(np.abs(J - Jo.reshape(-1))) <= J_RTOL * max(np.max(np.abs(Jo)), 1e-300)
                else:
                    assert rel_err(J, out.reshape(-1)) <= J_RTOL


# ---------------------------------------------------------------------------
# 7. sdp_p2p_broadcast
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("backend", BACKENDS)
def test_broadcast_pieces(product, backend):
    """pieces of 0, 1, 255, 257 and 592*256 + 3 values (more than one pass of the grid-stride loop
    of the capped grid) at offset 0, at an odd offset and at the end: every other rank receives
    exactly the piece, the source's buffer and everything outside the piece stay as they were, and
    every rank's epoch advances, for n = 0 too"""
    from stodynprog_b200 import _cabi
    sv = _toy(_Api(product, backend), 1, "plain")
    eng = sv.engine
    n_grid, N, k = 400001, 3, 1
    em = Ranks(eng, N, n_grid)
    rng = np.random.default_rng(9)
    src_data = rng.standard_normal(n_grid)
    for n in (0, 1, 255, 257, 592 * 256 + 3):
        for offset in (0, 12345, n_grid - n):
            s = (n + offset) % N                                   # the source rank
            for r in range(N):
                em.J[r][k].fill_(-1000.0 - r)
            em.J[s][k].copy_(eng.to_device(src_data))
            for r in range(N):
                src = em.J[r][k]
                m = n if r == s else 0                             # (every rank calls it, the others with n = 0)
                rc = eng.lib.sdp_p2p_broadcast(_ptr(src), offset if r == s else 0, m,
                                               ctypes.byref(em.peers[r][k, False]), eng.stream)
                _cabi.check(rc, "sdp_p2p_broadcast")
                em.published(r)
            em.wait_all()
            for r in range(N):
                got = _np(em.J[r][k])
                if r == s:
                    assert np.array_equal(got.view(np.int64), src_data.view(np.int64)), (n, offset)
                else:
                    want = np.full(n_grid, -1000.0 - r)
                    want[offset:offset + n] = src_data[offset:offset + n]
                    assert np.array_equal(got.view(np.int64), want.view(np.int64)), (n, offset, r)


# ---------------------------------------------------------------------------
# barrier
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("N", [1, 2, 3, 8])
def test_barrier_in_both_orders(product, backend, N):
    """sdp_p2p_barrier of every rank, once in rank order and once in reverse order; before each
    round the host pre-writes, in the flag array of every rank, the flags of the ranks that come
    after it with exactly the epoch they will publish (so no barrier waits on a flag nobody wrote
    yet); afterwards every flag word holds what the kernels published"""
    from stodynprog_b200 import _cabi
    eng = _toy(_Api(product, backend), 1, "plain").engine
    em = Ranks(eng, N, 64)
    for order in (list(range(N)), list(range(N))[::-1]):
        e = em.calls[0] + 1
        for i, r in enumerate(order):
            for q in order[i + 1:]:
                em.flags[r][q] = e
        for i, r in enumerate(order):
            em.ready(r, e, skip_own=True)      # (its own flag is the first thing its kernel writes)
            _cabi.check(eng.lib.sdp_p2p_barrier(ctypes.byref(em.peers[r][0, True]), eng.stream), "sdp_p2p_barrier")
            em.calls[r] += 1
            em.check(flags=False)
        em.check()


# ---------------------------------------------------------------------------
# 8. the comparisons have teeth
# ---------------------------------------------------------------------------
@gpu
def test_missing_remote_stores_are_seen(product, monkeypatch):
    """with the library's wrong-results switch dbg_exchange = 1 (no stores into other ranks'
    buffers) a sweep of shards of columns leaves the peers' slabs at the sentinel on every rank,
    and the comparison of test_column_shards fails"""
    from stodynprog_b200.engine import Engine
    monkeypatch.setattr(Engine, "COLUMN_BANDS", "1")
    make = _maker(product, "cuda", "CF", "curtail_9")
    full = make()
    T_full = full.sweep_tables()
    shape = full._state_grid_shape
    n_grid, n_rows = int(np.prod(shape)), shape[0]
    n_cols = n_grid // n_rows
    J0 = np.random.default_rng(23).standard_normal(shape)
    (J_want, A_want), = _full_sweeps(full, J0)
    cuts = _col_cuts(T_full, 3, n_rows, n_cols)
    shards = _shards(make, cuts, "columns")
    em = Ranks(full.engine, 3, n_grid)
    em.load(0, J0)
    em.fill(1)
    lib = full.engine.lib
    try:
        lib.sdp_set_option(b"dbg_exchange", 1)
        _exchange(em, shards, 0, 1, True, n_cols, cuts)
    finally:
        lib.sdp_set_option(b"dbg_exchange", 0)
    em.wait_all()
    for r in range(3):
        own = np.zeros((n_rows, n_cols), dtype=bool)
        own[:, cuts[r]:cuts[r + 1]] = True
        own = own.reshape(-1)
        J, A = _np(em.J[r][1]), _np(em.A[r])
        assert _same_bits(J[own], J_want[own]) and np.array_equal(A[own], A_want[own]), r
        assert np.all(J[~own] == SENT_J) and np.all(A[~own] == SENT_A), r
    with pytest.raises(AssertionError):
        _check_ranks(em, shards, 1, True, J_want, A_want, n_cols, cuts)


# ---------------------------------------------------------------------------
# 9. refusals (CPU: nothing reaches the device) and the ctypes mirror of SdpPeers
# ---------------------------------------------------------------------------
def test_refusals_launch_nothing(product):
    """every p2p entry point refuses, with SDP_EINVAL and no launch: world 0 or 9, a rank outside
    the world, NULL flags / epoch / done / J, a negative state_begin, glob_cols < col_begin +
    n_cols, tables not in layout CF for the _cols combine, incomplete reference-state arguments"""
    from stodynprog_b200 import _cabi
    lib = _cabi.load_library()
    J = [np.zeros(16) for _ in range(2)]
    flags = [np.zeros(2, dtype=np.uint64) for _ in range(2)]
    ed = np.zeros(2, dtype=np.uint64)
    vp = lambda a: a.ctypes.data_as(ctypes.c_void_p)          # noqa: E731

    def peers(**kw):
        P = _cabi.SdpPeers()
        P.world, P.rank = 2, 0
        for q in range(2):
            P.J[q], P.flags[q] = J[q].ctypes.data, flags[q].ctypes.data
        P.epoch, P.done = ed.ctypes.data, ed.ctypes.data + 8
        for k, v in kw.items():
            if k in ("J", "flags"):
                getattr(P, k)[1] = v
            else:
                setattr(P, k, v)
        return P

    def tables(layout=_cabi.LAYOUT_COLUMN_FACTORED, n_cols=4):
        c = _cabi.SdpTables()
        c.W, c.expect, c.layout, c.n_states, c.n_cols, c.tiles_per_col, c.u_mask = 1, 1, layout, 0, n_cols, 1, 1
        return c

    grid = _cabi.SdpGrid()
    grid.d, grid.order[0], grid.smin[0], grid.smax[0] = 1, 16, 0.0, 1.0
    arg = np.zeros(16, dtype=np.int32)
    one = np.zeros(4)
    i1 = np.zeros(4, dtype=np.int32)

    def calls(P, names=None):
        T = tables()
        B = ctypes.byref
        todo = {
            "finalize_p2p": lambda: lib.sdp_sweep_finalize_p2p(B(T), None, None, vp(arg), B(P), 0, None),
            "finalize_p2p_cols": lambda: lib.sdp_sweep_finalize_p2p_cols(B(T), None, None, vp(arg), B(P), 8, 0, None),
            "wait": lambda: lib.sdp_p2p_wait(B(P), None),
            "partials_after": lambda: lib.sdp_sweep_partials_after(B(grid), B(T), vp(J[0]), None, None, B(P), None),
            "broadcast": lambda: lib.sdp_p2p_broadcast(vp(J[0]), 0, 4, B(P), None),
            "barrier": lambda: lib.sdp_p2p_barrier(B(P), None),
            "policy_eval_p2p": lambda: lib.sdp_policy_eval_p2p(B(grid), 1, 0, None, None, None, 0, None, 0, 0, 16,
                                                       vp(J[0]), B(P), None, None, None, None, None)}
        return dict((k, f()) for k, f in todo.items() if names is None or k in names)

    n0 = lib.sdp_launch_count()
    bad_peers = [(peers(world=0), b"world/rank"), (peers(world=9), b"world/rank"), (peers(rank=2), b"world/rank"),
                 (peers(rank=-1), b"world/rank"), (peers(flags=None), b"NULL flag"),
                 (peers(epoch=None), b"epoch/done"), (peers(done=None), b"epoch/done")]
    for P, msg in bad_peers:
        for name, rc in calls(P).items():
            assert rc == -1, (name, msg)
            assert msg in lib.sdp_last_error(), (name, msg, lib.sdp_last_error())
    # NULL J buffer of a peer: every entry point that stores into the peers refuses it
    for name, rc in calls(peers(J=None), ("finalize_p2p", "finalize_p2p_cols", "broadcast", "policy_eval_p2p")).items():
        assert rc == -1 and b"NULL J" in lib.sdp_last_error(), name
    B = ctypes.byref
    P = peers()
    assert lib.sdp_sweep_finalize_p2p(B(tables()), None, None, vp(arg), B(P), -1, None) == -1
    assert b"bad arguments" in lib.sdp_last_error()
    assert lib.sdp_policy_eval_p2p(B(grid), 1, 0, None, None, None, 0, None, 0, -1, 16, vp(J[0]), B(P),
                                   None, None, None, None, None) == -1
    assert lib.sdp_sweep_finalize_p2p_cols(B(tables(n_cols=4)), None, None, vp(arg), B(P), 3, 0, None) == -1
    assert lib.sdp_sweep_finalize_p2p_cols(B(tables(n_cols=4)), None, None, vp(arg), B(P), 8, 5, None) == -1
    assert lib.sdp_sweep_finalize_p2p_cols(B(tables(n_cols=4)), None, None, vp(arg), B(P), 8, -1, None) == -1
    assert b"bad arguments" in lib.sdp_last_error()
    assert lib.sdp_sweep_finalize_p2p_cols(B(tables(_cabi.LAYOUT_STATE_MINOR_FACTORED)), None, None, vp(arg), B(P),
                                           8, 0, None) == -1
    assert b"not in layout CF" in lib.sdp_last_error()
    assert lib.sdp_p2p_broadcast(vp(J[0]), -1, 4, B(P), None) == -1
    assert lib.sdp_p2p_broadcast(vp(J[0]), 0, -1, B(P), None) == -1
    assert lib.sdp_p2p_broadcast(None, 0, 4, B(P), None) == -1
    for k in range(3):              # reference-state arguments: ref_cell given, one of the others missing
        a = [vp(one), vp(one), vp(one)]
        a[k] = None
        assert lib.sdp_policy_eval_p2p(B(grid), 1, 0, vp(one), None, None, 0, None, 0, 0, 16, vp(J[0]), B(P),
                                       vp(i1), a[0], a[1], a[2], None) == -1, k
        assert b"incomplete reference-state" in lib.sdp_last_error(), k
    assert lib.sdp_policy_eval_p2p(B(grid), 1, 0, None, None, None, 0, None, 0, 0, 16, vp(J[0]), B(P),
                                   vp(i1), vp(one), vp(one), vp(one), None) == -1         # (p NULL)
    assert lib.sdp_launch_count() == n0


def test_sdp_peers_layout_matches_the_header(tmp_path):
    """the ctypes mirror of SdpPeers: size and the offsets of J, flags, epoch, done and A, compiled
    against include/sdp_b200.h"""
    from stodynprog_b200 import _cabi
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler")
    src = tmp_path / "peers.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "sdp_b200.h"\n'
                   'int main(void){printf("%zu %zu %zu %zu %zu %zu %zu %d\\n", sizeof(SdpPeers), '
                   'offsetof(SdpPeers, J), offsetof(SdpPeers, flags), offsetof(SdpPeers, epoch), '
                   'offsetof(SdpPeers, done), offsetof(SdpPeers, A), offsetof(SdpPeers, rank), SDP_MAX_PEERS);'
                   'return 0;}\n')
    exe = tmp_path / "peers"
    subprocess.check_call([cc, "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = list(map(int, subprocess.check_output([str(exe)]).split()))
    P = _cabi.SdpPeers
    assert got == [ctypes.sizeof(P), P.J.offset, P.flags.offset, P.epoch.offset, P.done.offset, P.A.offset,
                   P.rank.offset, _cabi.SDP_MAX_PEERS]
