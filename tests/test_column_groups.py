"""Layout CF, group skipping (sdp_column_groups_build, option "col_groups"): the pruning column
sweep passes over whole groups of K controls that provably lose for every lane, from a 16-byte
summary per (item, group, lane), without reading their (x,u) stream.  The results must be those
of the full sweep, bit for bit.

CPU: a group skip (tablebuild.column_group_skip, twin of the device code) implies the per-control
skip (column_prune_skip) of every member, on random and adversarial groups; the window minima
against brute force.  GPU: the device summaries against the numpy builder; group skipping on, off
and no pruning at all on every column case over several sweeps with NaN / inf in J, for every
launch shape, with ties everywhere, on config #5, after a rebuild in recycled buffers and with no
summary registered."""
import ctypes

import numpy as np
import pytest

from test_column_prune import _kernel_value
from test_parity import COLUMN_CASES, _Api, _column_case, _same_bits

gpu = pytest.mark.gpu


def _row_bound(R, q, p):
    """(m(q), A(q)) as the pre-pass computes them (column_bound)"""
    m, a = np.float64(0.0), np.float64(0.0)
    with np.errstate(invalid="ignore", over="ignore"):
        for w in range(R.shape[1]):
            x, y = R[q, w], R[q + 1, w]
            m = m + np.float64(p[w]) * np.fmin(x, y)
            a = np.fmax(a, np.fmax(abs(x), abs(y)))
    if np.isnan(R[q]).any() or np.isnan(R[q + 1]).any():
        a = np.float64(np.nan)
    return m, a


def _column(R, p):
    """m, Acol of a table (rows x W): the last row's bound is the sentinel (0, NaN)"""
    rows = R.shape[0]
    mb = [_row_bound(R, q, p) for q in range(rows - 1)]
    m = np.array([x[0] for x in mb] + [0.0])
    A = np.array([x[1] for x in mb])
    acol = np.float64(np.nan) if np.isnan(A).any() else np.float64(A.max())
    return m, acol


def _group_skips(summary, Wm, L, acol, sum_p, best):
    from stodynprog_b200.tablebuild import column_group_skip, group_row_bound
    gmin, gabs, qlo, qhi = summary
    if qlo == 0xffff:
        return True                       # no live control: the lane needs nothing
    if qhi == 0xffff:
        return False
    m_lo = group_row_bound(Wm, L, qlo, qhi)
    return m_lo is not None and column_group_skip(gmin, gabs, m_lo, acol, sum_p, best)


def test_group_skip_implies_member_skip():
    """whenever the group test says "skip" for a lane, column_prune_skip skips each of its live
    controls, and the value the kernel computes is strictly greater than the best"""
    from stodynprog_b200.tablebuild import column_group_summary, column_prune_skip, window_minima
    rng = np.random.default_rng(20261022)
    specials = [np.nan, np.inf, -np.inf, 2.0 ** 1000, -(2.0 ** 1000), 2.0 ** 999, 1e300]
    lam_out = [np.nextafter(0.0, -1.0), np.nextafter(1.0, 2.0), np.nan]
    n_groups = n_skip = 0
    spans = {"below": 0, "within": 0, "above": 0}
    for _ in range(600):
        W = int(rng.choice([1, 3, 5, 9]))
        rows = int(rng.integers(6, 60))
        L = int(rng.choice([1, 2, 4, 8, 16]))
        p = rng.random(W)
        p = p / p.sum()
        sum_p = 0.0
        for x in p:
            sum_p += x
        R = rng.standard_normal((rows, W)).cumsum(axis=0) * 0.1 + np.linspace(0, 3, rows)[:, None]
        if rng.random() < 0.05:
            R[rng.integers(rows), rng.integers(W)] = rng.choice(specials)
        m, acol = _column(R, p)
        Wm = window_minima(m, L)
        K = int(rng.choice([8, 16]))
        live = rng.random(K) < 0.9
        q0 = int(rng.integers(0, rows - 1))
        width = int(rng.choice([0, 1, L - 1, L, 2 * L - 1, 2 * L, 3 * L]))
        q = np.clip(q0 + rng.integers(0, width + 1, K), 0, rows - 1)
        g = rng.standard_normal(K) * (10.0 ** rng.integers(-2, 3))
        lam = rng.random(K)
        if rng.random() < 0.1:
            g[rng.integers(K)] = rng.choice(specials)
        if rng.random() < 0.1:
            lam[rng.integers(K)] = rng.choice(lam_out)
        summary = column_group_summary(g, lam, q, live, rows)
        if summary[0] == 0xffff or summary[3] == 0xffff:
            pass
        else:
            span = summary[3] - summary[2] + 1
            spans["below" if span < L else ("within" if span <= 2 * L else "above")] += 1
        vals = [_kernel_value(g[k], lam[k], R[q[k]], R[min(q[k] + 1, rows - 1)], p, True)
                for k in range(K) if live[k] and q[k] <= rows - 2]
        for best in [np.inf, -np.inf, np.nan, 0.0] + [v for v in vals[:2]] + \
                [np.nextafter(min(vals), -np.inf) if vals else 0.0, (min(vals) - 0.5) if vals else 1.0]:
            best = np.float64(best)
            n_groups += 1
            if not _group_skips(summary, Wm, L, acol, sum_p, best) or summary[2] == 0xffff:
                continue
            n_skip += 1
            for k in range(K):
                if live[k]:
                    assert column_prune_skip(g[k], lam[k], R[q[k]], R[q[k] + 1], p, True, best), (k, best)
                    v = _kernel_value(g[k], lam[k], R[q[k]], R[q[k] + 1], p, True)
                    assert not np.isnan(v) and v > best
    assert n_skip > n_groups // 20                       # not vacuous
    assert min(spans.values()) > 50, spans               # spans below L, within [L, 2L] and above


def test_group_skip_refuses():
    """no group skip with a NaN / inf in the column's rows, |g| + A beyond 2^1000, a best of +inf or
    NaN, an ineligible group, or a span beyond 2L"""
    from stodynprog_b200.tablebuild import column_group_skip, column_group_summary, window_minima
    assert column_group_skip(1.0, 1.0, 0.0, 1.0, 1.0, 0.0)
    assert not column_group_skip(1.0, 1.0, 0.0, np.nan, 1.0, 0.0)
    assert not column_group_skip(1.0, np.inf, 0.0, 1.0, 1.0, 0.0)
    assert not column_group_skip(1.0, 2.0 ** 1000, 0.0, 1.0, 1.0, 0.0)
    assert not column_group_skip(1.0, 1.0, 0.0, 1.0, 1.0, np.inf)
    assert not column_group_skip(1.0, 1.0, 0.0, 1.0, 1.0, np.nan)
    live = np.ones(4, dtype=bool)
    q = np.array([3, 4, 4, 5])
    assert column_group_summary([1, 2, 3, 4], [0, .5, 1, .2], q, live, 10)[3] == 5
    for g, lam, qq in (([1, 2, np.nan, 4], [0, .5, 1, .2], q), ([1, 2, 3, 4], [0, .5, 1 + 1e-16 * 3, .2], q),
                       ([1, 2, 3, 4], [0, -5e-324, 1, .2], q), ([1, 2, 3, 4], [0, .5, 1, .2], q + 4)):
        assert column_group_summary(g, lam, qq, live, 10)[3] == 0xffff
    assert column_group_summary([1, 2], [.5, .5], [1, 2], [False, False], 10)[2] == 0xffff
    m = np.arange(40.0)
    Wm = window_minima(m, 4)
    assert _group_skips((1.0, 1.0, 0, 7), Wm, 4, 1.0, 1.0, -100.0)
    assert not _group_skips((1.0, 1.0, 0, 8), Wm, 4, 1.0, 1.0, -100.0)      # span 9 > 2L


def test_window_minima_brute_force():
    """Wm against brute force; the two-window bound is the exact minimum for spans in [L, 2L] and a
    lower bound below L"""
    from stodynprog_b200.tablebuild import group_row_bound, window_minima
    rng = np.random.default_rng(3)
    for _ in range(200):
        rows = int(rng.integers(2, 90))
        m = rng.standard_normal(rows)
        if rng.random() < 0.3:
            m[rng.integers(rows)] = np.nan
        m[-1] = 0.0                               # the sentinel row takes no part
        for L in (1, 2, 4, 8, 32):
            Wm = window_minima(m, L)
            for qq in range(rows - 1):
                assert _same_bits(Wm[qq], np.fmin.reduce(m[qq:min(qq + L, rows - 1)]))
            for _ in range(20):
                qlo = int(rng.integers(0, rows - 1))
                qhi = int(rng.integers(qlo, rows - 1))
                b = group_row_bound(Wm, L, qlo, qhi)
                if qhi - qlo >= 2 * L:
                    assert b is None
                    continue
                exact = np.fmin.reduce(m[qlo:qhi + 1])
                if qhi - qlo + 1 >= L:
                    assert _same_bits(b, exact)
                elif not np.isnan(exact):
                    assert b <= exact


def _numpy_summaries(T, rows, stride0, K):
    """the summaries of tables T (host copies), [item][group][lane] -> (gmin, gabs, qlo, qhi)"""
    from stodynprog_b200.tablebuild import column_group_summary
    items = np.frombuffer(T.items.cpu().numpy().tobytes(), dtype=__import__("stodynprog_b200")._cabi.ITEM_DTYPE)
    cell, lam, g = T.cell.cpu().numpy(), T.lam.cpu().numpy(), T.g.cpu().numpy()
    U = T.U_dev.cpu().numpy()
    inv = 1.0 / float(stride0)
    out = []
    for it in items:
        Us = U[int(it["state"]) * 32:int(it["state"]) * 32 + 32]
        n = int(it["u_count"])
        for g0 in range(0, n, K):
            for lane in range(32):
                uu = np.arange(g0, min(g0 + K, n))
                o = int(it["entry_base"]) + uu * 32 + lane
                live = int(it["u_begin"]) + uu < Us[lane]
                q = np.rint(cell[o].astype(np.float64) * inv).astype(np.int64)
                out.append(column_group_summary(g[o], lam[o], q, live, rows))
    return out


def test_numpy_summaries_on_model_tables(product):
    """the numpy builder on tables of the numpy model: every live control of a group lies within
    its summary, and the padding lanes have none"""
    sv = _column_case(_Api(product, "model", "state_minor", "auto", "on"), "ar1_w3")
    sv.column_hoist = "on"
    T = sv.sweep_tables()
    assert T.layout_name == "column_factored" and T.col_groups is None      # (built for the GPU only)
    rows, stride0 = sv._state_grid_shape[0], int(np.prod(sv._state_grid_shape[1:]))
    S = _numpy_summaries(T, rows, stride0, 8)
    live = [s for s in S if s[2] != 0xffff]
    assert 0 < len(live) < len(S)
    assert all(s[2] <= s[3] for s in live)
    assert any(s[3] != 0xffff for s in live)


# ---------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------
def _solver(product, which):
    sv = _column_case(_Api(product, "cuda", "state_minor", "auto", "on"), which)
    sv.column_hoist, sv.column_pairs = "on", "off"
    return sv


def _vi(sv, J, prune, groups):
    lib = sv.engine.lib
    lib.sdp_set_option(b"col_prune", prune)
    lib.sdp_set_option(b"col_groups", groups)
    try:
        return sv.value_iteration(J, report_time=False)
    finally:
        lib.sdp_set_option(b"col_prune", 1)
        lib.sdp_set_option(b"col_groups", 1)


def _kernel_name(sv):
    from stodynprog_b200 import _cabi
    return _cabi.last_kernel()


@gpu
@pytest.mark.parametrize("which", COLUMN_CASES)
def test_groups_are_bit_identical(product, which):
    """groups on, groups off and no pruning, each on its own cached tables, over 5 sweeps with NaN /
    inf injected into J, then every launch shape of the pruning test"""
    svs = [_solver(product, which) for _ in range(3)]
    J0 = np.random.default_rng(11).standard_normal(svs[0]._state_grid_shape)
    for sweep in range(5):
        (Jr, pr), (Jo, po), (Jg, pg) = _vi(svs[0], J0, 0, 0), _vi(svs[1], J0, 1, 0), _vi(svs[2], J0, 1, 1)
        assert svs[2].last_tables.col_groups is not None
        assert "groups" in _kernel_name(svs[2]), _kernel_name(svs[2])
        for J, pol in ((Jo, po), (Jg, pg)):
            assert _same_bits(Jr, J), sweep
            assert np.array_equal(pr, pol, equal_nan=True), sweep
        J0 = Jr.copy()
        if sweep == 2:
            J0.reshape(-1)[::7] = np.nan
            J0.reshape(-1)[3::11] = np.inf
    col, lib = svs[2], svs[2].engine.lib
    try:
        Jr, pr = _vi(svs[0], J0, 0, 0)
        for threads, ub, pf, pre in ((128, 1, 1, 1), (256, 2, 1, 0), (512, 1, 2, 0), (96, 2, 2, 2),
                                     (640, 2, 1, 2), (768, 1, 2, 0), (704, 1, 1, 2), (768, 2, 1, 3),
                                     (640, 1, 2, 3), (64, 2, 2, 3)):
            lib.sdp_set_option(b"col_threads", threads)
            lib.sdp_set_option(b"col_ub", ub)
            lib.sdp_set_option(b"col_pf", pf)
            lib.sdp_set_option(b"col_prepass", pre)
            lib.sdp_set_option(b"col_dynamic", (threads // 32) % 2)
            for _ in range(2):
                J2, p2 = _vi(col, J0, 1, 1)
                assert _same_bits(Jr, J2), (threads, ub, pf, pre)
                assert np.array_equal(pr, p2, equal_nan=True), (threads, ub, pf, pre)
    finally:
        lib.sdp_set_option(b"col_threads", 0)
        lib.sdp_set_option(b"col_ub", 2)
        lib.sdp_set_option(b"col_pf", 2)
        lib.sdp_set_option(b"col_prepass", 3)
        lib.sdp_set_option(b"col_dynamic", 1)


@gpu
def test_groups_with_ties_everywhere(product):
    """J constant along axis 0: whole runs of controls tie exactly"""
    svs = [_solver(product, "ar1_w9") for _ in range(3)]
    dims = svs[0]._state_grid_shape
    J0 = np.broadcast_to(np.random.default_rng(5).standard_normal((1,) + dims[1:]), dims).copy()
    for _ in range(4):
        (Jr, pr), (Jo, po), (Jg, pg) = _vi(svs[0], J0, 0, 0), _vi(svs[1], J0, 1, 0), _vi(svs[2], J0, 1, 1)
        assert _same_bits(Jr, Jo) and _same_bits(Jr, Jg)
        assert np.array_equal(pr, po, equal_nan=True) and np.array_equal(pr, pg, equal_nan=True)


def _device_summaries(T):
    """the registered buffer of T, decoded like the numpy builder's output"""
    from stodynprog_b200 import _cabi
    n_items = T.n_items
    raw = T.col_groups.cpu().numpy()
    off = 256 + ((8 * n_items + 15) & ~15)
    ent = raw[off:].view(np.float64).reshape(-1, 2)
    y = ent[:, 1].view(np.uint64)
    gabs = (y & np.uint64(0xffffffff)).astype(np.uint32).view(np.float32).astype(np.float64)
    qlo = ((y >> np.uint64(32)) & np.uint64(0xffff)).astype(np.int64)
    qhi = (y >> np.uint64(48)).astype(np.int64)
    assert _cabi.SDP_ABI_VERSION == 10
    return ent[:, 0], gabs, qlo, qhi


@gpu
@pytest.mark.parametrize("which", ["ar1_w9", "ar1_w4", "searev", "curtail"])
def test_device_summaries_match_numpy(product, which):
    sv = _solver(product, which)
    T = sv.sweep_tables()
    K, L = ctypes.c_int32(), ctypes.c_int32()
    assert sv.engine.lib.sdp_column_groups_info(T.col_groups_id, ctypes.byref(K), ctypes.byref(L)) == 0
    assert K.value == 8 and L.value >= 1
    rows, stride0 = sv._state_grid_shape[0], int(np.prod(sv._state_grid_shape[1:]))
    want = _numpy_summaries(T, rows, stride0, K.value)
    gmin, gabs, qlo, qhi = _device_summaries(T)
    assert len(want) <= len(gmin)
    for k, (wg, wa, wl, wh) in enumerate(want):
        assert (qlo[k], qhi[k]) == (wl, wh), k
        if wl != 0xffff:
            assert _same_bits(gmin[k], wg) and _same_bits(gabs[k], wa), k


@gpu
def test_groups_config5(product):
    """config #5 over 4 device-resident sweeps: J and argmin bit for bit with groups on, off and no
    pruning; groups are passed over and their warp steps count as skipped"""
    import torch
    import workloads as wl
    sv = wl.storage_ar1_large(_Api(product, "cuda")).solver
    T = sv.sweep_tables()
    assert T.layout_name == "column_factored" and T.col_groups is not None
    eng, lib = sv.engine, sv.engine.lib
    n = int(np.prod(sv._state_grid_shape))
    J0 = np.random.default_rng(0).standard_normal(sv._state_grid_shape)
    res = {}
    try:
        for prune, groups in ((0, 0), (1, 0), (1, 1)):
            lib.sdp_set_option(b"col_prune", prune)
            lib.sdp_set_option(b"col_groups", groups)
            lib.sdp_set_option(b"col_prune_stats", 1)
            T.part_idx.fill_(-1)
            J_prev, J_new = eng.J_pair(n)
            eng.begin_call(n)
            eng.upload_J(J0, J_prev)
            seq = []
            for _ in range(4):
                eng.sweep(T, J_prev, J_new)
                J_prev, J_new = J_new, J_prev
                torch.cuda.synchronize()
                seq.append((J_prev.clone().cpu().numpy(), T.argmin.cpu().numpy().copy()))
            c = [ctypes.c_int64() for _ in range(4)]
            assert lib.sdp_col_prune_counts(ctypes.byref(c[0]), ctypes.byref(c[1])) == 0
            assert lib.sdp_col_group_counts(ctypes.byref(c[2]), ctypes.byref(c[3])) == 0
            res[(prune, groups)] = (seq, [x.value for x in c])
    finally:
        lib.sdp_set_option(b"col_prune", 1)
        lib.sdp_set_option(b"col_groups", 1)
        lib.sdp_set_option(b"col_prune_stats", 0)
    for key in ((1, 0), (1, 1)):
        for (Ja, Aa), (Jb, Ab) in zip(res[(0, 0)][0], res[key][0]):
            assert np.array_equal(Ja.view(np.int64), Jb.view(np.int64)) and np.array_equal(Aa, Ab)
    off, on = res[(1, 0)][1], res[(1, 1)][1]
    assert off[2] == 0 and on[2] > 0 and 0 < on[3] <= on[2]
    assert on[0] == off[0] and 0 < on[1] <= on[0]          # the same warp steps, group skips among them


def _scaled_cost(cost):
    """-3 c + 1, with the five positional arguments of the storage cost (the system checks the arity)"""
    def scaled(E, P_mis, P_sto, P_cur, innov):
        return -3.0 * np.asarray(cost(E, P_mis, P_sto, P_cur, innov)) + 1.0
    return scaled


@gpu
def test_groups_after_rebuild_in_recycled_buffers(product):
    """a new cost, tables rebuilt into the buffers of the old ones (as a per-instant recursion
    does): the summaries of the old tables are gone, the new ones describe the new entries"""
    sv = _solver(product, "ar1_w5")
    ref = _solver(product, "ar1_w5")
    eng = sv.engine
    J0 = np.random.default_rng(9).standard_normal(sv._state_grid_shape)
    _vi(sv, J0, 1, 1)
    T = sv.last_tables
    ptrs = (T.cell.data_ptr(), T.g.data_ptr())
    for s in (sv, ref):
        assert len(s.sys._dyn_args) == 5
        s.sys.cost = _scaled_cost(s.sys.cost)
        s.clear_tables()
    T2 = eng.build_sweep_tables(sv, None, reuse=T)
    assert T2 is T and (T.cell.data_ptr(), T.g.data_ptr()) == ptrs and T.col_groups is not None
    sv._table_cache = {sv._cache_key(None): T2}
    T2.probe_fingerprint = sv._probe_fingerprint(None)
    for _ in range(3):
        Jr, pr = _vi(ref, J0, 0, 0)
        Jg, pg = _vi(sv, J0, 1, 1)
        assert sv.last_tables is T2 and "groups" in _kernel_name(sv)
        assert _same_bits(Jr, Jg) and np.array_equal(pr, pg, equal_nan=True)
        J0 = Jr.copy()


@gpu
def test_groups_not_registered(product):
    """tables whose summary was released (or never built) sweep without group skipping, with the
    same results"""
    from stodynprog_b200.tablebuild import release_column_groups
    sv, ref = _solver(product, "ar1_w9"), _solver(product, "ar1_w9")
    J0 = np.random.default_rng(4).standard_normal(sv._state_grid_shape)
    _vi(sv, J0, 1, 1)
    release_column_groups(sv.last_tables)
    for _ in range(3):
        Jr, pr = _vi(ref, J0, 0, 0)
        Jg, pg = _vi(sv, J0, 1, 1)
        assert "groups" not in _kernel_name(sv) and "prune" in _kernel_name(sv)
        assert _same_bits(Jr, Jg) and np.array_equal(pr, pg, equal_nan=True)
        J0 = Jr.copy()
