"""Host-side API tests (CPU suite).  The SysDescription tests read like the
reference's own (stodynprog/tests/test_stodynprog.py); the rest covers the
solver's host logic and the C-ABI library (load + exported symbols only: no
compute call is made without a GPU)."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

import stodynprog_b200 as sdp
from stodynprog_b200 import _cabi, tabulate as tb
from stodynprog_b200.sysdesc import _zero_cost, _enforce_sig_len
from conftest import ROOT, golden


# --- mirror of reference tests/test_stodynprog.py ---------------------------
def test_zero_cost():
    assert _zero_cost() == 0.
    assert _zero_cost(1) == 0.
    assert _zero_cost(1, 2) == 0.
    assert _zero_cost(1, 2, 3) == 0.


def test_enforce_sig_len():
    def f0():
        pass

    def f1(x):
        pass

    def f2(x, y):
        pass
    arg0, arg1, arg2 = [], ['x'], ['x', 'y']
    wp = False
    assert _enforce_sig_len(f0, arg0, wp)
    for f, bad in ((f0, arg1), (f0, arg2), (f1, arg0), (f1, arg2), (f2, arg1), (f2, arg0)):
        with pytest.raises(ValueError):
            _enforce_sig_len(f, bad, wp)
    assert _enforce_sig_len(f1, arg1, wp)
    assert _enforce_sig_len(f2, arg2, wp)
    with pytest.raises(ValueError) as e:
        _enforce_sig_len(f1, arg2, wp)
    assert e.value.args[0] == "'f1' should accept 2 args (x, y), not 1"   # reference test :58

    def f1p(x, **params):
        pass
    assert _enforce_sig_len(f1p, arg1, with_params=True)
    with pytest.raises(ValueError):
        _enforce_sig_len(f1p, arg1, with_params=False)
    with pytest.raises(ValueError):
        _enforce_sig_len(f1, arg1, with_params=True)


class TestSysDescription:
    def setup_method(self):
        self.sys110 = sdp.SysDescription((1, 1, 0), stationnary=True, name='sys110')
        self.sys111 = sdp.SysDescription((1, 1, 1), stationnary=True, name='sys111')

    def test_attributes(self):
        assert self.sys111.stationnary
        assert self.sys111.stochastic
        assert not self.sys110.stochastic
        assert self.sys111.name == 'sys111'

    def test_dyn_function(self):
        def dyn3(my_state, my_control, my_perturb):
            pass
        self.sys111.dyn = dyn3
        assert self.sys111.state == ['my_state']
        assert self.sys111.control == ['my_control']
        assert self.sys111.perturb == ['my_perturb']

        def dyn2(x, u):
            pass

        def dyn4(x, y, u, w):
            pass
        with pytest.raises(ValueError):
            self.sys111.dyn = dyn2
        with pytest.raises(ValueError):
            self.sys111.dyn = dyn4

    def test_print_summary(self, capsys):
        self.sys111.print_summary()
        out = capsys.readouterr().out
        assert 'Dynamical system "sys111" description' in out
        assert 'stationnary, stochastic' in out

    def test_time_dependent_and_params(self):
        s = sdp.SysDescription((1, 1), stationnary=False, params={'a': 1})

        def dyn(k, x, u, **p):
            return (x + u,)
        s.dyn = dyn
        assert s.state == ['x'] and s.control == ['u'] and s.perturb == []

        def box(k, x, **p):
            return ((0, 1),)
        s.control_box = box
        with pytest.raises(ValueError):
            s.cost = lambda k, x, u: 0      # missing **params
        with pytest.raises(ValueError):
            sdp.SysDescription((1,))

    def test_perturb_laws(self):
        import scipy.stats as stats
        self.sys111.perturb_laws = [stats.norm()]
        assert self.sys111.perturb_types == ['continuous']
        self.sys111.perturb_laws = [stats.poisson(2)]
        assert self.sys111.perturb_types == ['discrete']
        with pytest.raises(ValueError):
            self.sys111.perturb_laws = []
        with pytest.raises(ValueError):
            self.sys111.perturb_laws = [object()]

    def test_terminal_cost(self):
        with pytest.raises(ValueError):
            self.sys111.terminal_cost = lambda x, y: 0
        self.sys111.terminal_cost = lambda x: x
        assert self.sys111.terminal_cost(3) == 3


# --- DPSolver host logic -------------------------------------------------------
def test_discretize_and_reference_state():
    import workloads as wl
    sv = wl.storage_ar1(sdp).solver
    assert sv._state_grid_shape == (41, 61)
    assert sv._state_ref_ind == (20, 30)
    assert sv._state_ref == (sv.state_grid[0][20], sv.state_grid[1][30])
    assert np.allclose(sum(sv.perturb_proba[0]), 1.0)
    g = sv.state_grid_full
    assert g[0].shape == (41, 61) and g[1][3, 7] == sv.state_grid[1][7]
    with pytest.raises(AssertionError):
        sv.discretize_state(0, 1, 3)
    with pytest.raises(AssertionError):
        sv.discretize_perturb(0, 1)


def test_discrete_pmf_must_sum_to_one():
    import workloads as wl
    sv = wl.inventory(sdp).solver
    assert list(sv.perturb_proba[0]) == [0.2, 0.4, 0.3, 0.1]
    with pytest.raises(AssertionError):
        sv.discretize_perturb(0, 2, 3)       # misses the mass at w = 3


def test_control_grids_match_port(port):
    import workloads as wl
    import itertools
    a = wl.storage_ar1(sdp).solver
    b = wl.storage_ar1(port).solver
    for x_k in itertools.islice(itertools.product(*a.state_grid), 0, 2501, 37):
        ga, da = a.control_grids(x_k)
        gb, db = b.control_grids(x_k)
        assert da == db
        for u, v in zip(ga, gb):
            assert np.array_equal(u, v)
    ga, da = a.control_grids((0.0, 0.0))
    assert da == (4001, 1) and ga[1][0] == 0.0


def test_control_axis_values_equals_linspace():
    rng = np.random.default_rng(0)
    for _ in range(300):
        lo = rng.normal() * 10.0 ** rng.integers(-3, 4)
        hi = lo + abs(rng.normal()) * 10.0 ** rng.integers(-3, 4)
        n = int(rng.integers(2, 400))
        ref = np.linspace(lo, hi, n)
        idx = np.arange(n)
        got = tb.control_axis_values(np.full(n, lo), np.full(n, hi), np.full(n, n), idx)
        assert np.array_equal(got, ref)
    # degenerate: zero width, and the single centre point
    assert np.array_equal(tb.control_axis_values([1.0] * 3, [1.0] * 3, [3] * 3, [0, 1, 2]), np.linspace(1., 1., 3))
    assert tb.control_axis_values([0.0], [0.0], [1], [0])[0] == 0.0
    assert tb.control_axis_values([2.0], [3.0], [1], [0])[0] == 2.5


def test_batched_control_box_scan():
    """a box function written with element-wise numpy is scanned in one call and
    agrees with the per-state scan; the reference's `np.max((a, b))` style does
    not vectorise and must be rejected (the engine then scans per state)"""
    grid = [np.linspace(0, 10, 23), np.linspace(-4, 4, 17)]
    steps = (0.031, 0.1)

    def box_vec(E, P):
        return ((np.maximum(-E / 1.0, -4.0), np.minimum((10 - E) / 1.0, 4.0)), (0, 0))

    def box_ref_style(E, P):
        return ((np.max((-E / 1.0, -4.0)), np.min(((10 - E) / 1.0, 4.0))), (0, 0))

    class S(object):
        control = ['a', 'b']
        params = {}
    S.control_box = staticmethod(box_vec)
    n = 23 * 17
    tab = tb.scan_control_boxes_batched(S, steps, grid, 5, n - 3)
    ref = tb.scan_control_boxes(S, steps, tb.state_tuples(grid, 5, n - 3))
    assert tab is not None
    assert np.array_equal(tab.lo, ref.lo) and np.array_equal(tab.hi, ref.hi)
    assert np.array_equal(tab.npts, ref.npts) and tab.npts.max() > 100
    S.control_box = staticmethod(box_ref_style)
    assert tb.scan_control_boxes_batched(S, steps, grid, 0, n) is None

    # a box that vectorises but to the wrong thing (a global reduction) is caught by the check
    def box_wrong(E, P):
        return ((np.max(-E), np.min(10 - E)), (0, 0))
    S.control_box = staticmethod(box_wrong)
    assert tb.scan_control_boxes_batched(S, steps, grid, 0, n) is None


def test_rebalance_bounds():
    from stodynprog_b200.engine import rebalance_bounds, partition_by_weight
    U = np.full(8000, 200)
    b0 = partition_by_weight(U + 1, 4)
    assert b0 == [0, 2000, 4000, 6000, 8000]
    # balanced within tolerance, or a missing time: nothing moves
    assert rebalance_bounds(U, b0, [1.0, 1.01, 0.99, 1.0]) is None
    assert rebalance_bounds(U, b0, [1.0, 0.0, 1.0, 1.0]) is None
    # slab 1 is 20 % slower: it shrinks, the others grow, and the estimated times equalise
    t = np.array([1.0, 1.2, 1.0, 1.0])
    b1 = rebalance_bounds(U, b0, t)
    assert b1[0] == 0 and b1[-1] == 8000 and b1 == sorted(b1)
    assert b1[2] - b1[1] < 2000 < b1[1] - b1[0]
    density = np.repeat(t / 2000.0, 2000)
    est = [density[b1[r]:b1[r + 1]].sum() for r in range(4)]
    assert max(est) / min(est) < 1.002
    assert max(est) < 1.06          # was 1.2 before the re-cut


def test_make_items_cuts_units_into_equal_runs():
    from stodynprog_b200.engine import make_items
    U = np.array([140, 1, 512, 513, 129, 4, 0, 256])
    off = np.arange(len(U)) * 100000
    for chunk in (4, 32, 128, 512):
        items, begin = make_items(U, chunk, off, 9 * 32, off // 2, 32, None)
        assert begin[0] == 0 and begin[-1] == len(items)
        for k, u in enumerate(U):
            it = items[begin[k]:begin[k + 1]]
            assert len(it) == -(-u // chunk)
            if u == 0:
                continue
            # the runs tile [0, u) in order, none is empty, none exceeds the chunk
            assert it["u_begin"][0] == 0 and np.all(it["u_begin"][1:] == np.cumsum(it["u_count"])[:-1])
            assert it["u_count"].sum() == u and it["u_count"].min() >= 1 and it["u_count"].max() <= chunk
            assert np.all(it["u_begin"] % 4 == 0)
            # equal lengths up to the rounding to a multiple of 4
            assert it["u_count"].max() - it["u_count"].min() <= 4 * len(it) + 3
            assert np.all(it["state"] == k)
            assert np.all(it["entry_base"] == off[k] + it["u_begin"].astype(np.int64) * 9 * 32)
            assert np.all(it["g_base"] == off[k] // 2 + it["u_begin"].astype(np.int64) * 32)
    items, _ = make_items(np.array([140]), 128, [0], 1, [0], 1, np.array([140]))
    assert list(items["u_count"]) == [72, 68] and list(items["Upad"]) == [140, 140]


def test_column_piece_cuts():
    """pieces of columns for the host results of layout CF: a partition of the columns in sweep
    order, never an empty piece, cuts on multiples of the CTA count where that is close"""
    from hypothesis import given, settings, strategies as st
    from stodynprog_b200.tablebuild import column_piece_cuts
    # config #5 on a B200: 500 equal columns, 148 CTAs
    even = np.arange(501, dtype=float)
    assert column_piece_cuts(even, (0.3, 0.3, 0.3, 0.1), 148) == [0, 148, 296, 444, 500]
    assert column_piece_cuts(even, (0.5, 0.25, 0.15, 0.1), 148) == [0, 296, 375, 450, 500]
    assert column_piece_cuts(even, (0.5, 0.25, 0.15, 0.1), 0) == [0, 250, 375, 450, 500]
    assert column_piece_cuts(even[:3], (0.3, 0.3, 0.3, 0.1), 148) == [0, 1, 2]
    assert column_piece_cuts(even[:2], (0.5, 0.5), 148) == [0, 1]

    @settings(max_examples=300, deadline=None)
    @given(st.lists(st.floats(0.0, 50.0), min_size=1, max_size=700),
           st.lists(st.floats(0.01, 1.0), min_size=1, max_size=6), st.integers(0, 200))
    def prop(weights, fractions, n_ctas):
        csum = np.concatenate([[0.0], np.cumsum(weights)])
        cuts = column_piece_cuts(csum, tuple(fractions), n_ctas)
        assert cuts[0] == 0 and cuts[-1] == len(weights)
        assert all(a < b for a, b in zip(cuts, cuts[1:]))
        assert len(cuts) - 1 <= len(fractions)
    prop()


def test_pick_item_chunk():
    from stodynprog_b200.engine import pick_item_chunk, ITEMS_TARGET
    # plenty of units: keep the long runs
    assert pick_item_chunk(np.full(40000, 256), 32) == 512
    # one eighth of the large grid (a rank of an 8-GPU run): runs are cut until the launch
    # is several waves of warps long
    c = pick_item_chunk(np.full(3907, 256), 32)
    assert c == 64 and ((256 + c - 1) // c) * 3907 >= ITEMS_TARGET
    # tiny problems stop at the floor
    assert pick_item_chunk(np.full(10, 100), 128) == 128


def test_interp_on_state_errors():
    import workloads as wl
    sv = wl.storage_ar1(sdp, n_E=5, n_P=6).solver
    with pytest.raises(ValueError) as e:
        sv.interp_on_state(np.zeros((6, 5)))
    assert e.value.args[0] == 'array `A` should be of shape (5, 6), not (6, 5)'
    f = sv.interp_on_state(np.zeros((5, 6)))
    assert f.ndim == 2 and f.values.shape == (1, 30)
    import pickle
    g = pickle.loads(pickle.dumps(f))           # stays picklable like the reference's
    assert np.array_equal(g._xmax, f._xmax) and np.array_equal(g.values, f.values)


def test_print_summary_matches_notebook(capsys):
    """examples/howto storage-AR1.ipynb cell 8 output"""
    import workloads as wl
    sv = wl.storage_ar1(sdp).solver
    sv.print_summary()
    out = capsys.readouterr().out
    assert '* state space discretized on a 41x61 points grid' in out
    assert 'yields [4,001 to 8,001] possible values (6,342.5 on average)' in out
    assert 'control combinations: [4,001 to 8,001] possible values (6,342.5 on average)' in out


def test_partition_by_weight():
    from stodynprog_b200.engine import partition_by_weight
    w = np.array([1, 1, 1, 1, 10, 1, 1, 1, 1, 1], dtype=float)
    b = partition_by_weight(w, 2)
    assert b[0] == 0 and b[-1] == 10 and b == sorted(b)
    rng = np.random.default_rng(0)
    w = rng.integers(129, 257, size=100000).astype(float)
    for world in (2, 4, 8):
        b = partition_by_weight(w, world)
        loads = [w[b[r]:b[r + 1]].sum() for r in range(world)]
        assert len(b) == world + 1 and b[0] == 0 and b[-1] == len(w)
        assert max(loads) / (w.sum() / world) < 1.001
    assert partition_by_weight([], 4) == [0, 0, 0, 0, 0]
    assert partition_by_weight([5.0], 4)[-1] == 1


# --- the C ABI -----------------------------------------------------------------
def _header_symbols():
    txt = open(os.path.join(ROOT, "include", "sdp_b200.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(sdp_[a-z0-9_]+)\s*\(", txt)))


def test_library_loads_and_exports_every_declared_symbol(product):
    lib = _cabi.load_library()
    declared = _header_symbols()
    assert len(declared) >= 14
    for name in declared:
        assert hasattr(lib, name), name
        assert name in _cabi.SIGNATURES, "binding missing for " + name
    assert sorted(_cabi.SIGNATURES) == declared
    assert lib.sdp_version() == _cabi.SDP_ABI_VERSION
    out = subprocess.run(["nm", "-D", "--defined-only", _cabi.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (sdp_[a-z0-9_]+)", out))
    assert set(declared) <= exported


def test_struct_layouts_match_the_header(tmp_path):
    """numpy / ctypes mirrors vs the C compiler's view of include/sdp_b200.h"""
    src = tmp_path / "layout.c"
    src.write_text('''
#include <stdio.h>
#include <stddef.h>
#include "sdp_b200.h"
int main(void) {
  printf("%zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(SdpStateDesc), offsetof(SdpStateDesc, src),
         offsetof(SdpStateDesc, cs), offsetof(SdpStateDesc, ws), offsetof(SdpStateDesc, npts),
         offsetof(SdpStateDesc, U), offsetof(SdpStateDesc, Upad), sizeof(SdpItem));
  printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu %lld\\n", sizeof(SdpTables), offsetof(SdpTables, p), offsetof(SdpTables, n_items),
         offsetof(SdpTables, U), sizeof(SdpGrid), offsetof(SdpTables, p_host), offsetof(SdpTables, n_cols),
         offsetof(SdpTables, seg_begin), offsetof(SdpTables, n_segs), offsetof(SdpTables, col_table),
         (long long)SDP_COLUMN_PITCH(2000, 9) * 1000 + (long long)SDP_COLUMN_PITCH(7, 4));
  return 0; }''')
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    l1, l2 = subprocess.run([str(exe)], capture_output=True, text=True).stdout.strip().splitlines()
    D = _cabi.STATE_DESC_DTYPE
    assert [int(x) for x in l1.split()] == [D.itemsize, D.fields["src"][1], D.fields["cs"][1],
                                            D.fields["ws"][1], D.fields["npts"][1], D.fields["U"][1],
                                            D.fields["Upad"][1], _cabi.ITEM_DTYPE.itemsize]
    T = _cabi.SdpTables
    assert [int(x) for x in l2.split()] == [ctypes.sizeof(T), T.p.offset, T.n_items.offset, T.U.offset,
                                            ctypes.sizeof(_cabi.SdpGrid), T.p_host.offset, T.n_cols.offset,
                                            T.seg_begin.offset, T.n_segs.offset, T.col_table.offset,
                                            _cabi.column_pitch(2000, 9) * 1000 + _cabi.column_pitch(7, 4)]
    hdr = open(os.path.join(ROOT, "include", "sdp_b200.h")).read()
    for name in ("SDP_ABI_VERSION", "SDP_LAYOUT_COLUMN_FACTORED", "SDP_FACTORED_MAX_W_REG"):
        val = int(re.search(r"#define %s (\d+)" % name, hdr).group(1))
        assert val == getattr(_cabi, name.replace("SDP_LAYOUT_", "LAYOUT_").replace("SDP_FACTORED", "FACTORED"))
    assert _cabi.COLUMN_MAX_SMEM_BYTES == 200 * 1024 and "SDP_COLUMN_MAX_SMEM_BYTES (200 * 1024)" in hdr


def test_column_order_and_row_aligned_bounds():
    """layout CF walks a slab of whole rows band by band, column by column, every column
    of a band padded to whole tiles of 32 rows; slab boundaries are moved to whole rows"""
    from stodynprog_b200.engine import column_order, row_aligned, item_run_ends, column_segments
    order, valid, tiles, tile_begin, tile_col, _ = column_order(70 * 5, 5)
    assert tiles == [3] and tile_begin == [0, 15] and len(order) == 5 * 96 and valid.sum() == 350
    assert sorted(order[valid]) == list(range(350))              # every state exactly once
    assert list(tile_col) == [0, 0, 0, 1, 1, 1, 2, 2, 2, 3, 3, 3, 4, 4, 4]
    o = order.reshape(5, 96)
    v = valid.reshape(5, 96)
    for c in range(5):
        assert list(o[c, :70]) == [r * 5 + c for r in range(70)]   # lane <-> row of the column
        assert np.all(o[c, 70:] == 69 * 5 + c) and not v[c, 70:].any() and v[c, :70].all()
    order, valid, tiles, tile_begin, tile_col, _ = column_order(64 * 3, 3)
    assert tiles == [2] and valid.all() and len(order) == 192
    # two bands: rows 0..39 (2 tiles per column, 24 padding lanes) and 40..69 (1 tile, 2 padding lanes)
    order, valid, tiles, tile_begin, tile_col, pos_row = column_order(70 * 5, 5, [0, 40, 70])
    assert pos_row is None and tiles == [2, 1] and tile_begin == [0, 10, 15] and len(order) == 32 * 15
    assert sorted(order[valid]) == list(range(350))
    assert list(tile_col) == [0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 0, 1, 2, 3, 4]
    assert list(order[:40]) == [r * 5 for r in range(40)] and not valid[40:64].any()
    band1 = order[320:].reshape(5, 32)
    assert list(band1[2, :30]) == [r * 5 + 2 for r in range(40, 70)]
    with pytest.raises(AssertionError):
        column_order(70 * 5, 5, [0, 40, 60])
    # two rows per lane: rows r, r+1 share a lane where pair_ok[r]; a lone row gets a padding
    # position beside it; every band is padded to whole PAIRS of tiles (64 positions)
    from stodynprog_b200.engine import pair_positions
    ok = np.ones(69, dtype=bool)
    ok[[4, 9, 10]] = False                     # rows 4|5, 9|10, 10|11 must not share a lane
    pr = pair_positions(0, 40, ok)
    assert list(pr[:14]) == [0, 1, 2, 3, 4, -1, 5, 6, 7, 8, 9, -1, 10, -1] and len(pr) == 64
    assert sorted(pr[pr >= 0]) == list(range(40)) and np.all(pr[0::2] >= 0) == (pr[0::2] >= 0).all()
    for a, b in zip(pr[0::2], pr[1::2]):
        assert b == -1 or (b == a + 1 and ok[a])
    order, valid, tiles, tile_begin, tile_col, pos_row = column_order(70 * 5, 5, [0, 40, 70], ok)
    assert tiles == [2, 2] and tile_begin == [0, 10, 20] and len(order) == 64 * 10
    assert sorted(order[valid]) == list(range(350)) and len(pos_row) == 2
    assert list(pos_row[0]) == list(pr) and sorted(pos_row[1][pos_row[1] >= 0]) == list(range(30))
    band1 = order[320:].reshape(5, 64)
    assert np.array_equal(band1[3][pos_row[1] >= 0], (40 + pos_row[1][pos_row[1] >= 0]) * 5 + 3)
    assert list(item_run_ends([3, 3, 3, 4, 9, 9])) == [3, 3, 3, 4, 6, 6]
    assert list(item_run_ends([])) == [] and list(item_run_ends([7])) == [1]
    seg = column_segments(np.array([10, 10, 10, 10, 30, 10]), 3)
    assert seg[0] == 0 and seg[-1] == 6 and len(seg) == 4 and np.all(np.diff(seg) >= 0)
    assert list(column_segments(np.array([5, 5]), 148)) == [0, 1, 2]
    assert row_aligned([0, 103, 251, 350], 5) == [0, 105, 250, 350]
    assert row_aligned([0, 2, 3, 350], 5) == [0, 0, 5, 350]
    assert row_aligned([0, 349, 350], 5) == [0, 350, 350]


def test_parallel_control_box_scan(monkeypatch):
    """the per-state control_box scan on forked workers: same boxes and grid sizes, bit for
    bit; None (serial scan takes over) when a worker fails; used by the table build of large
    single-rank grids"""
    import workloads as wl
    from stodynprog_b200 import tabulate as tb
    from stodynprog_b200.engine import Engine
    from fake_lib import FakeLib
    sv = wl.storage_ar1(sdp, n_E=23, n_P=7, steps=(0.3, 0.1), _test_lib=FakeLib()).solver
    n = 23 * 7
    serial = tb.scan_control_boxes(sv.sys, sv.control_steps, tb.state_tuples(sv.state_grid, 5, n - 3))
    par = tb.scan_control_boxes_parallel(sv.sys, sv.control_steps, sv.state_grid, 5, n - 3, None, procs=3)
    assert par is not None
    assert np.array_equal(par.lo.view(np.int64), serial.lo.view(np.int64))
    assert np.array_equal(par.hi.view(np.int64), serial.hi.view(np.int64))
    assert np.array_equal(par.npts, serial.npts)
    assert tb.state_tuples_at(sv.state_grid, 17, 60) == tb.state_tuples(sv.state_grid, 17, 60)
    assert tb.scan_control_boxes_parallel(sv.sys, sv.control_steps, sv.state_grid, 0, n, None, procs=1) is None

    def bad_box(E, P_mis):
        raise RuntimeError("box function failing in a worker")
    good = sv.sys.control_box
    sv.sys._control_box = bad_box            # (bypasses the signature check of the setter)
    try:
        assert tb.scan_control_boxes_parallel(sv.sys, sv.control_steps, sv.state_grid, 0, n, None, procs=2) is None
    finally:
        sv.sys._control_box = good
    # the table build takes the parallel scan above its size threshold: same tables
    J0 = np.random.default_rng(0).standard_normal((23, 7))
    J_a, pol_a = sv.value_iteration(J0, report_time=False)
    calls = []
    real = tb.scan_control_boxes_parallel
    monkeypatch.setattr(tb, "scan_control_boxes_parallel", lambda *a, **k: calls.append(1) or real(*a, **k))
    monkeypatch.setattr(Engine, "SCAN_PARALLEL_MIN_STATES", 10)
    monkeypatch.setattr(Engine, "SCAN_PROCS", 2)
    sv2 = wl.storage_ar1(sdp, n_E=23, n_P=7, steps=(0.3, 0.1), _test_lib=FakeLib()).solver
    J_b, pol_b = sv2.value_iteration(J0, report_time=False)
    assert calls and np.array_equal(J_a, J_b) and np.array_equal(pol_a, pol_b)


def test_control_box_scan_by_axes():
    """box functions that ignore some state variables (np.max((a, b)) on scalars: not
    vectorisable) are scanned once per distinct box and checked on sample states: same table,
    bit for bit; a box that reads every axis, or one whose dependence hides from the probe but not
    from the check, gives None (per-state scan)"""
    import workloads as wl
    from fake_lib import FakeLib
    sv = wl.storage_ar1(sdp, n_E=90, n_P=70, steps=(0.3, 0.1), _test_lib=FakeLib()).solver
    n = 90 * 70
    calls = [0]
    good = sv.sys.control_box

    def counting(E, P_mis):
        calls[0] += 1
        return good(E, P_mis)
    sv.sys._control_box = counting
    fast = tb.scan_control_boxes_by_axes(sv.sys, sv.control_steps, sv.state_grid, 100, n - 50)
    n_calls = calls[0]
    sv.sys._control_box = good
    serial = tb.scan_control_boxes(sv.sys, sv.control_steps, tb.state_tuples(sv.state_grid, 100, n - 50))
    assert fast is not None and n_calls < n // 2
    assert np.array_equal(fast.lo.view(np.int64), serial.lo.view(np.int64))
    assert np.array_equal(fast.hi.view(np.int64), serial.hi.view(np.int64))
    assert np.array_equal(fast.npts, serial.npts)

    def both_axes(E, P_mis):
        return ((-E - 1., P_mis + 10.), (0, 0))
    sv.sys._control_box = both_axes
    assert tb.scan_control_boxes_by_axes(sv.sys, sv.control_steps, sv.state_grid, 0, n) is None

    def hidden(E, P_mis):           # depends on P_mis only in a corner the axis probe does not visit
        lo, hi = good(E, P_mis)[0]
        return ((lo, hi + (1.0 if (E > 9.9 and P_mis > 3.9) else 0.0)), (0, 0))
    sv.sys._control_box = hidden
    assert tb.scan_control_boxes_by_axes(sv.sys, sv.control_steps, sv.state_grid, 0, n) is None
    sv.sys._control_box = good


def test_batched_tabulation_checks_every_chunk():
    """a cost that is not element-wise over the state axis in ONE region of the state space only
    must be caught although the first chunk verifies: the batched mode is abandoned"""
    import workloads as wl
    from fake_lib import FakeLib
    prob = wl.storage_ar1(sdp, n_E=64, n_P=8, steps=(0.5, 0.1), _test_lib=FakeLib())
    sv = prob.solver
    good = sv.sys.cost

    def sneaky(E, P_mis, P_sto, P_cur, innov):
        g = good(E, P_mis, P_sto, P_cur, innov)
        if np.ndim(E) > 0 and np.max(E) > 9.:       # chunks holding the top of the E range only
            g = g + 1e-3 * np.mean(E)               # depends on the whole chunk
        return g
    sv.sys._cost = sneaky
    seen = []
    real = tb.tabulate_states_batched

    def small_chunks(*a, **k):
        k["chunk_states"] = 128
        try:
            return real(*a, **k)
        except tb.BatchedMismatch:
            seen.append("mismatch")
            raise
    tb.tabulate_states_batched = small_chunks
    try:
        T = sv.sweep_tables()
    finally:
        tb.tabulate_states_batched = real
    assert seen and T.tabulate_mode == "per_state"


@pytest.mark.parametrize("layout", ["auto", "control_minor"])
def test_host_threads_give_the_same_tables(layout):
    """DPSolver.host_threads: chunks evaluated on worker threads, staged in order by the caller:
    the same tables, bit for bit, the calls really made off the calling thread, and a chunk that
    fails its check still ends the batched mode"""
    import threading
    import workloads as wl
    from fake_lib import FakeLib
    real = tb.tabulate_states_batched

    def small_chunks(*a, **k):
        k["chunk_states"] = 96
        return real(*a, **k)

    def tables(threads, cost_wrapper=None):
        prob = wl.storage_ar1(sdp, n_E=70, n_P=33, steps=(0.3, 0.1), _test_lib=FakeLib())
        sv = prob.solver
        sv.table_layout = layout
        sv.host_threads = threads
        if cost_wrapper:
            sv.sys._cost = cost_wrapper(sv.sys.cost)
        tb.tabulate_states_batched = small_chunks
        try:
            return sv.sweep_tables(), sv
        finally:
            tb.tabulate_states_batched = real

    names = set()

    def noting(cost):
        def f(*a):
            if np.ndim(a[0]) > 0:
                names.add(threading.current_thread().name)
            return cost(*a)
        return f
    (T1, sv1), (T4, sv4) = tables(1), tables(4, noting)
    assert T1.tabulate_mode == T4.tabulate_mode == "batched"
    assert any(n.startswith("sdp-tabulate") for n in names)
    assert T1.n_entries == T4.n_entries
    for name in ("cell", "lam", "g"):       # (the allocations end in uninitialised padding)
        a, b = getattr(T1, name).numpy()[:T1.n_entries], getattr(T4, name).numpy()[:T1.n_entries]
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), name
    J0 = np.random.default_rng(3).standard_normal(sv1._state_grid_shape)
    (J1, p1), (J4, p4) = sv1.value_iteration(J0), sv4.value_iteration(J0)
    assert np.array_equal(J1.view(np.int64), J4.view(np.int64)) and np.array_equal(p1, p4)
    assert tables("auto")[0].tabulate_mode == "batched"

    def sneaky(cost):
        def f(E, *a):
            g = cost(E, *a)
            return g + 1e-3 * np.mean(E) if (np.ndim(E) > 0 and np.max(E) > 9.) else g
        return f
    assert tables(4, sneaky)[0].tabulate_mode == "per_state"
    with pytest.raises(ValueError):
        tables(0)


def test_cached_tables_follow_the_callables(port):
    """The reference calls dyn / cost / control_box afresh in every sweep, so a change of a
    global or closure variable they read takes effect at once (its doc/example_inventory.py cost
    reads h, p, c).  Cached tables are re-validated on probe states and rebuilt."""
    import workloads as wl
    from fake_lib import FakeLib
    price = [1.0]

    def build(api, **kw):
        prob = wl.inventory(api, **kw)
        base = prob.sys.cost
        prob.sys.cost = lambda x, u, w: base(x, u, w) * price[0]
        return prob.solver
    sv, ora = build(sdp, _test_lib=FakeLib()), build(port)
    J0 = np.zeros(10)
    for p_now in (1.0, 1.0, 2.5, 2.5):
        price[0] = p_now
        J, pol = sv.value_iteration(J0, report_time=False)
        Jo, polo = ora.value_iteration(J0)
        assert np.array_equal(pol, polo) and np.allclose(J, Jo, rtol=1e-12, atol=0)
        Js, pols, _ = sv.solve_value_iteration(J_zero=J0, max_iter=1)
        assert np.array_equal(pols, polo)
    # the control-box scan is re-checked too
    cap = [10]
    sv2, ora2 = wl.inventory(sdp, _test_lib=FakeLib()).solver, wl.inventory(port).solver
    for s_ in (sv2, ora2):
        s_.sys._control_box = lambda x: ((0, cap[0]),)
    sv2.cache_tables = False
    for c_now in (10, 4):
        cap[0] = c_now
        J, pol = sv2.value_iteration(J0 - np.arange(10.), report_time=False)
        Jo, polo = ora2.value_iteration(J0 - np.arange(10.))
        assert np.array_equal(pol, polo) and np.allclose(J, Jo, rtol=1e-12, atol=0)


@pytest.mark.parametrize("d", [1, 2, 3, 4])
def test_host_interpolation_routine_is_bit_exact(product, d):
    """sdp_interp_host / sdp_interp_host_f32 (the latency path for a handful of points: host
    pointers, no launch) against the outputs of the reference's own compiled Cython routine on
    the adversarial fixture points (outside the grid, +-3e9, +-1e300, +-inf, NaN), fp64 and fp32"""
    G = golden("interp_kat.npz")
    lib = _cabi.load_library()
    smin, smax, orders = G["d%d_smin" % d], G["d%d_smax" % d], G["d%d_orders" % d]
    g = _cabi.SdpGrid()
    g.d = d
    for k in range(d):
        g.order[k], g.smin[k], g.smax[k] = int(orders[k]), float(smin[k]), float(smax[k])
    for dtype, fn, want in ((np.float64, lib.sdp_interp_host, G["d%d_out" % d]),
                            (np.float32, lib.sdp_interp_host_f32, G["d%d_out_f32" % d])):
        values = np.ascontiguousarray(G["d%d_values" % d], dtype=dtype)
        s = np.ascontiguousarray(G["d%d_s" % d], dtype=dtype)
        out = np.empty((values.shape[0], s.shape[1]), dtype=dtype)
        rc = fn(ctypes.byref(g), values.shape[0], values.ctypes.data_as(ctypes.c_void_p), s.shape[1],
                s.ctypes.data_as(ctypes.c_void_p), out.ctypes.data_as(ctypes.c_void_p))
        assert rc == 0
        bits = np.int64 if dtype == np.float64 else np.int32
        same = (out.view(bits) == want.view(bits)) | (np.isnan(out) & np.isnan(want))
        assert same.all(), (dtype, int((~same).sum()))


def test_no_cpu_fallback(product):
    """without a GPU the product refuses to run; without the library it says so"""
    import torch
    import workloads as wl
    if not torch.cuda.is_available():
        sv = wl.inventory(sdp).solver
        with pytest.raises(_cabi.SdpLibraryError):
            sv.value_iteration(np.zeros(10), report_time=False)
    with pytest.raises(_cabi.SdpLibraryError):
        _cabi.load_library("/nonexistent/libsdp_b200.so")


def test_product_does_not_import_the_oracle():
    """the oracle is test infrastructure: nothing under stodynprog_b200/ refers to it"""
    pkg = os.path.join(ROOT, "stodynprog_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), f
                assert "liboracle" not in txt and "sdp_oracle" not in txt, f


# the kernel families that divide: the IEEE division sequence is built from FMAs, which is
# exact by construction.  Every other kernel promises an exact operation order (bit-identity to
# the oracle or to a numpy model, the rounding margin of DESIGN.md section 4) and must have none.
FMA_ALLOWED = {"k_build_tables", "k_build_tables_tiled", "k_build_factored", "k_build_factored_tiled",
               "k_cell_setup", "k_interp", "k_policy_values", "k_combine_column", "k_combine_column_small"}


def _kernel_family(fn):
    """the kernel's name without template arguments or parameter types (_Z<len><name>...)"""
    m = re.match(r"_Z(\d+)(\w+)", fn)
    return m.group(2)[:int(m.group(1))] if m else fn


def test_sass_has_no_fma_in_sweep_kernels(product):
    """the parity contract forbids contraction: no kernel may contain DFMA / FFMA except the
    division-bearing families of FMA_ALLOWED; a new kernel with FMA fails with its name"""
    res = subprocess.run(["cuobjdump", "-sass", _cabi.LIB_PATH], capture_output=True, text=True)
    if res.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    fn, bad, families = None, {}, set()
    for line in res.stdout.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            fn = m.group(1)
            families.add(_kernel_family(fn))
        elif fn and re.search(r"\b[DF]FMA", line) and _kernel_family(fn) not in FMA_ALLOWED:
            bad[fn] = bad.get(fn, 0) + 1
    assert not bad, bad
    # (not vacuous: the kernels that promise an exact order are all in the library)
    assert {"k_sweep_tiled", "k_policy_eval", "k_sub_scalar", "k_first_passage", "k_fwd_rows", "k_chain_sample",
            "k_column_table", "k_supnorm_diff"} <= families
    assert "UBLKCP" in res.stdout      # the TMA-fed variant is built (bulk async copies)
