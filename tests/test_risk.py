"""Risk-averse Bellman backups: the nested mean-CVaR operator (MeanCVaR, sdp_sweep_risk_partials,
sdp_policy_eval_risk[_p2p] of include/sdp_b200.h).

- The numpy twin (oracle/risk_port.py) against a textbook CVaR (Rockafellar-Uryasev: the
  minimum over t of t + E[(v - t)^+] / beta) on random values and probabilities with ties,
  zero-probability nodes, +-inf and NaN; its translation invariance and monotonicity; weight 0
  is the ordered expectation bit for bit.
- Argument checks, and that risk=None never reaches a risk entry point.
- Table choice: a risk sweep runs on layout A dense tables, kept beside the expectation's.
- CPU suite ("model"): the host code drives numpy models of the risk entry points
  (RiskFakeLib) against the port with the risk backup, for all five solver methods.
- GPU suite ("cuda"): the kernels against the port bit for bit (every d, both W buckets, NaN /
  inf in J), weight 0 against risk=None, optimality and monotonicity in the weight, on the
  benchmark configurations.
"""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from fake_lib import FakeLib, _arr, _grid
from oracle import risk_port as rp
from stodynprog_b200 import _cabi

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---------------------------------------------------------------------------
# the twin
# ---------------------------------------------------------------------------
def textbook_cvar(v, p, beta):
    """min over t of t + E[(v - t)^+] / beta (finite v), in exact-enough float"""
    live = p > 0
    v, p = v[live], p[live]
    best = np.inf
    for t in v:
        best = min(best, t + np.sum(p * np.maximum(v - t, 0.0)) / beta)
    return best


def _random_case(rng, n, W, ties=False, zeros=False):
    V = rng.standard_normal((n, W))
    if ties:
        V = np.round(V * 2) / 2
        V[:, ::3] = -0.0
    p = rng.random(W)
    if zeros:
        p[rng.random(W) < 0.3] = 0.0
        p[0] = max(p[0], 0.1)
    return V, p / p.sum()


@pytest.mark.parametrize("W", [1, 2, 5, 9, 16])
@pytest.mark.parametrize("alpha", [0.0, 0.3, 0.9, 0.99])
def test_twin_against_textbook_cvar(W, alpha):
    rng = np.random.default_rng(W * 100 + int(alpha * 100))
    for ties in (False, True):
        for zeros in (False, True):
            V, p = _random_case(rng, 50, W, ties, zeros)
            consts = rp.risk_constants(alpha, 1.0)
            got = rp.risk_values(V, p, consts)
            beta = consts[1]
            want = np.array([textbook_cvar(V[i], p, beta) for i in range(len(V))])
            # the walk stops at mass beta of a total that may round below 1: compare loosely
            assert np.allclose(got, want, rtol=1e-9, atol=1e-9 * np.max(np.abs(V)))


def test_twin_nonfinite_values():
    p = np.array([0.2, 0.3, 0.5])
    c = rp.risk_constants(0.5, 0.5)
    V = np.array([[1.0, np.nan, 0.0],          # NaN anywhere: C = NaN
                  [np.inf, 0.0, 1.0],          # +inf in the tail
                  [-np.inf, 0.0, 1.0],         # -inf below the tail: C finite, E = -inf
                  [1.0, 2.0, np.inf]])
    r = rp.risk_values(V, p, c)
    assert np.isnan(r[0])
    assert r[1] == np.inf
    assert r[2] == -np.inf
    assert r[3] == np.inf
    # -inf inside the tail of mass 1 (alpha = 0); with weight 1, E*0 is NaN when E is infinite
    assert rp.risk_values(np.array([[-np.inf, 1.0]]), np.array([0.5, 0.5]), rp.risk_constants(0.0, 0.5))[0] == -np.inf
    assert np.isnan(rp.risk_values(np.array([[-np.inf, 1.0]]), np.array([0.5, 0.5]), rp.risk_constants(0.0, 1.0))[0])
    # a NaN node of probability 0 still makes C NaN; with weight 0, rho = E*1 + NaN*0 = NaN
    assert np.isnan(rp.risk_values(np.array([[np.nan, 1.0]]), np.array([0.0, 1.0]), rp.risk_constants(0.5, 0.0))[0])


def test_twin_tie_order_and_zero_mass_nodes():
    # ties go to the lower w first; a node of probability 0 is skipped even at the top
    p = np.array([0.0, 0.25, 0.25, 0.5])
    V = np.array([[9.0, 1.0, 1.0, 0.0]])
    c = rp.risk_constants(0.75, 1.0)            # beta = 0.25: the tail is node 1
    assert rp.risk_values(V, p, c)[0] == 1.0
    c = rp.risk_constants(0.6, 1.0)             # beta = 0.4: node 1 whole, 0.15 of node 2
    assert rp.risk_values(V, p, c)[0] == (0.0 + 1.0 * 0.25 + 1.0 * (0.4 - 0.25)) * (1.0 / 0.4)


def test_twin_weight_zero_is_ordered_expectation():
    rng = np.random.default_rng(5)
    V, p = _random_case(rng, 200, 9, ties=True, zeros=True)
    E = np.zeros(len(V))
    for w in range(9):
        E = E + V[:, w] * p[w]
    r = rp.risk_values(V, p, rp.risk_constants(0.7, 0.0))
    assert np.array_equal(r, E)


def test_twin_translation_invariance_and_monotonicity():
    rng = np.random.default_rng(7)
    V, p = _random_case(rng, 300, 9, ties=True, zeros=True)
    c = rp.risk_constants(0.8, 0.6)
    r = rp.risk_values(V, p, c)
    for shift in (1.0, -3.5, 100.0):
        assert np.allclose(rp.risk_values(V + shift, p, c), r + shift, rtol=1e-12, atol=1e-12 * 100)
    bump = np.abs(rng.standard_normal(V.shape)) * (rng.random(V.shape) < 0.3)
    assert np.all(rp.risk_values(V + bump, p, c) >= r - 1e-12 * (1 + np.abs(r)))


# ---------------------------------------------------------------------------
# arguments
# ---------------------------------------------------------------------------
def test_mean_cvar_validation(product):
    M = product.MeanCVaR
    for a, w in ((1.0, 0.5), (-0.1, 0.5), (0.5, 1.1), (0.5, -0.1), (float("nan"), 0.5), (0.5, float("nan"))):
        with pytest.raises(ValueError):
            M(a, w)
    r = M(0.9, 0.25)
    with pytest.raises(AttributeError):
        r.alpha = 0.5
    assert r.constants() == (1.0 / (1.0 - 0.9), 1.0 - 0.9, 0.75, 0.25)
    assert M(0.9, 0.25) == r and hash(M(0.9, 0.25)) == hash(r)


def test_sdprisk_layout_matches_header(tmp_path):
    src = tmp_path / "off.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "sdp_b200.h"\n'
                   'int main(void){printf("%zu %zu %zu %zu %zu %d\\n", sizeof(SdpRisk), '
                   'offsetof(SdpRisk, inv_beta), offsetof(SdpRisk, beta), offsetof(SdpRisk, w_mean), '
                   'offsetof(SdpRisk, w_cvar), SDP_RISK_MAX_W); return 0;}\n')
    exe = tmp_path / "off"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    R = _cabi.SdpRisk
    assert out == [ctypes.sizeof(R), R.inv_beta.offset, R.beta.offset, R.w_mean.offset, R.w_cvar.offset,
                   _cabi.RISK_MAX_W]


# ---------------------------------------------------------------------------
# numpy model of the risk entry points
# ---------------------------------------------------------------------------
def _consts(rref):
    r = rref._obj
    return r.inv_beta, r.beta, r.w_mean, r.w_cvar


class RiskFakeLib(FakeLib):
    def __init__(self):
        super().__init__()
        self.risk_calls = 0

    def sdp_sweep_risk_partials(self, gref, tref, rref, J_prev, part_val, part_idx, stream):
        T = tref._obj
        assert T.layout in (_cabi.LAYOUT_CONTROL_MINOR, _cabi.LAYOUT_COLUMN_FACTORED) and T.W <= _cabi.RISK_MAX_W
        self.risk_calls += 1
        if not T.expect:
            return self.sdp_sweep_partials(gref, tref, J_prev, part_val, part_idx, stream)
        if T.layout == _cabi.LAYOUT_COLUMN_FACTORED:
            return self._column_risk(gref, T, rref, J_prev, part_val, part_idx)
        d, smin, smax, orders = _grid(gref)
        J = _arr(J_prev, int(np.prod(orders)), ctypes.c_double)
        strides = np.concatenate([np.cumprod(orders[::-1])[::-1][1:], [1]]).astype(np.int64)
        items = np.frombuffer((ctypes.c_uint8 * (T.n_items * _cabi.ITEM_DTYPE.itemsize))
                              .from_address(T.items), dtype=_cabi.ITEM_DTYPE)
        p = _arr(T.p, T.W, ctypes.c_double)
        pv = _arr(part_val, T.n_items, ctypes.c_double)
        pi = _arr(part_idx, T.n_items, ctypes.c_int32)

        def lerp(c, lam):
            def rec(base, k):
                if k == d:
                    return J[base]
                return (1 - lam[k]) * rec(base, k + 1) + lam[k] * rec(base + strides[k], k + 1)
            return rec(c, 0)

        for n_it, it in enumerate(items):
            cnt, ub, Upad = int(it["u_count"]), int(it["u_begin"]), int(it["Upad"])
            V = np.zeros((cnt, T.W))
            with np.errstate(invalid="ignore"):
                for w in range(T.W):
                    off = int(it["entry_base"]) + w * Upad
                    c = _arr(T.cell + 4 * off, cnt, ctypes.c_int32).astype(np.int64)
                    lam = [_arr(T.lam + 8 * (k * T.lam_plane + off), cnt, ctypes.c_double) for k in range(d)]
                    g0 = int(it["g_base"]) + (w * Upad if T.g_per_w else 0)
                    V[:, w] = _arr(T.g + 8 * g0, cnt, ctypes.c_double) + lerp(c, lam)
                rho = rp.risk_values(V, p, _consts(rref))
            nan = np.isnan(rho)
            j = int(np.argmax(nan)) if nan.any() else int(np.argmin(rho))
            pv[n_it], pi[n_it] = rho[j], ub + j
        self.launches += 1
        return 0

    def _column_risk(self, gref, T, rref, J_prev, part_val, part_idx):
        """layout CF, one row per lane: the positions seg_begin[0] .. seg_begin[n_segs] of the work
        list; node values of the whole-grid lerp at cell_u + cell_w (the kernel reads the column
        tables of the pre-pass: the same bits)"""
        assert not T.col_pairs and T.col_table and T.seg_begin
        d, smin, smax, orders = _grid(gref)
        J = _arr(J_prev, int(np.prod(orders)), ctypes.c_double)
        strides = np.concatenate([np.cumprod(orders[::-1])[::-1][1:], [1]]).astype(np.int64)
        items = np.frombuffer((ctypes.c_uint8 * (T.n_items * _cabi.ITEM_DTYPE.itemsize))
                              .from_address(T.items), dtype=_cabi.ITEM_DTYPE)
        seg = _arr(T.seg_begin, T.n_segs + 1, ctypes.c_int64)
        order = _arr(T.item_order, T.n_items, ctypes.c_int64) if T.item_order else np.arange(T.n_items)
        p = _arr(T.p, T.W, ctypes.c_double)
        pv = _arr(part_val, T.n_items * 32, ctypes.c_double)
        pi = _arr(part_idx, T.n_items * 32, ctypes.c_int32)
        W, n_pos = T.W, (int(items["state"].max()) + 1) * 32
        Us = _arr(T.U, n_pos, ctypes.c_int32)

        def lerp(c, lam):
            def rec(base, k):
                if k == d:
                    return J[base]
                return (1 - lam[k]) * rec(base, k + 1) + lam[k] * rec(base + strides[k], k + 1)
            return rec(c, 0)

        for pos in range(int(seg[0]), int(seg[-1])):
            n_it = int(order[pos])
            it = items[n_it]
            cnt, ub, eb, tix = int(it["u_count"]), int(it["u_begin"]), int(it["entry_base"]), int(it["state"])
            cu = _arr(T.cell + 4 * eb, cnt * 32, ctypes.c_int32).astype(np.int64).reshape(cnt, 32)
            lu = [_arr(T.lam + 8 * eb, cnt * 32, ctypes.c_double).reshape(cnt, 32)]
            Gv = _arr(T.g + 8 * eb, cnt * 32, ctypes.c_double).reshape(cnt, 32)
            V = np.zeros((cnt, 32, W))
            with np.errstate(invalid="ignore"):
                for w in range(W):
                    f0 = ((tix // T.tiles_per_col) * T.tiles_per_col * W + w) * 32
                    cw = _arr(T.cell_w + 4 * f0, 1, ctypes.c_int32).astype(np.int64)[None, :]
                    lw = [_arr(T.lam_w + 8 * (j * T.lam_w_plane + f0), 1, ctypes.c_double)[None, :]
                          for j in range(d - 1)]
                    V[:, :, w] = Gv + lerp(cu + cw, self._merge(T, d, lu, lw))
                rho = rp.risk_values(V.reshape(-1, W), p, _consts(rref)).reshape(cnt, 32)
            for lane in range(32):
                n_ok = max(0, min(cnt, int(Us[tix * 32 + lane]) - ub))
                if n_ok == 0:
                    pv[n_it * 32 + lane], pi[n_it * 32 + lane] = np.inf, 2 ** 31 - 1
                    continue
                col = rho[:n_ok, lane]
                nan = np.isnan(col)
                j = int(np.argmax(nan)) if nan.any() else int(np.argmin(col))
                pv[n_it * 32 + lane], pi[n_it * 32 + lane] = col[j], ub + j
        self.launches += 1
        return 0

    def sdp_policy_eval_risk(self, gref, W, g_per_w, p, cell, lam, lam_plane, g, n_states, state_begin,
                             n_grid, J_a, J_b, n_iter, rel_dp, ref_index, hist, rref, stream):
        self.risk_calls += 1
        d, smin, smax, orders = _grid(gref)
        strides = np.concatenate([np.cumprod(orders[::-1])[::-1][1:], [1]]).astype(np.int64)
        P = _arr(p, W, ctypes.c_double)
        C = _arr(cell, W * n_states, ctypes.c_int32).astype(np.int64).reshape(W, n_states)
        L = [_arr(lam.value + 8 * k * lam_plane, W * n_states, ctypes.c_double).reshape(W, n_states)
             for k in range(d)]
        Gv = _arr(g, (W if g_per_w else 1) * n_states, ctypes.c_double).reshape(-1, n_states)
        A, B = _arr(J_a, n_grid, ctypes.c_double), _arr(J_b, n_grid, ctypes.c_double)
        H = _arr(hist, n_iter, ctypes.c_double) if rel_dp else None
        src, dst = A, B
        for it in range(n_iter):
            V = np.zeros((n_states, W))
            for w in range(W):
                lam_w = [L[k][w] for k in range(d)]

                def rec(base, k):
                    if k == d:
                        return src[base]
                    return (1 - lam_w[k]) * rec(base, k + 1) + lam_w[k] * rec(base + strides[k], k + 1)
                V[:, w] = Gv[w if g_per_w else 0] + rec(C[w], 0)
            dst[state_begin:state_begin + n_states] = rp.risk_values(V, P, _consts(rref))
            if rel_dp:
                H[it] = dst[ref_index]
                dst -= H[it]
            src, dst = dst, src
        self.launches += n_iter
        return 0


class _Api(object):
    def __init__(self, pkg, backend):
        self.pkg = pkg
        self.backend = backend
        self.SysDescription = pkg.SysDescription
        self.libs = []

    def DPSolver(self, sys, **kw):
        if self.backend == "model":
            kw["_test_lib"] = lib = RiskFakeLib()
            self.libs.append(lib)
        return self.pkg.DPSolver(sys, **kw)


@pytest.fixture(scope="module", params=[pytest.param("model", id="model"),
                                        pytest.param("cuda", marks=gpu, id="cuda")])
def api(request, product):
    return _Api(product, request.param)


@pytest.fixture(scope="module")
def cuda_api(product):
    return _Api(product, "cuda")


def same(a, b):
    """equal values, NaN where NaN (signed zeros compare equal)"""
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and bool(np.all((a == b) | (np.isnan(a) & np.isnan(b))))


def _toy(api, d, n_w=5, **kw):
    from test_parity import _toy as toy
    return toy(api, d, "w", n_w=n_w, **kw)


def _timedep(api):
    """1 state, 1 control, 1 perturbation on 7 nodes, a cost that depends on the instant"""
    import scipy.stats as stats

    def dyn(k, x, u, w):
        return (0.8 * x + 0.5 * u + 0.3 * w,)

    def box(k, x):
        return ((-1.0, 1.0),)

    def cost(k, x, u, w):
        return (1.0 + 0.1 * k) * x ** 2 + 0.2 * u ** 2 + 0.05 * k * w * u

    sys = api.SysDescription((1, 1, 1), stationnary=False, name='time-dependent toy')
    sys.dyn, sys.control_box, sys.cost = dyn, box, cost
    sys.perturb_laws = [stats.norm(0, 0.4)]
    sv = api.DPSolver(sys)
    sv.discretize_state(-2.0, 2.0, 17)
    sv.discretize_perturb(-1.0, 1.0, 7)
    sv.control_steps = (0.1,)
    return sv


RISK = (0.8, 0.5)
LAYOUT = {"A": "control_minor", "B": "state_minor", "AF": "control_minor_factored",
          "BF": "state_minor_factored", "CF": "column_factored"}


# ---------------------------------------------------------------------------
# host logic (model) and the same through the kernels (cuda)
# ---------------------------------------------------------------------------
def test_risk_none_never_calls_a_risk_entry_point(product):
    a = _Api(product, "model")
    sv = _toy(a, 2)
    J0 = np.random.default_rng(0).standard_normal(sv._state_grid_shape)
    J, pol = sv.value_iteration(J0, report_time=False)
    sv.solve_value_iteration(J0, max_iter=2)
    sv.eval_policy(pol, 3, report_time=False)
    assert a.libs[-1].risk_calls == 0
    sv.value_iteration(J0, report_time=False, risk=product.MeanCVaR(*RISK))
    assert a.libs[-1].risk_calls == 1


def test_risk_argument_errors(product):
    a = _Api(product, "model")
    sv = _toy(a, 1, n_w=17)
    J0 = np.zeros(sv._state_grid_shape)
    with pytest.raises(ValueError, match="W = 17.*16"):
        sv.value_iteration(J0, report_time=False, risk=product.MeanCVaR(*RISK))
    sv = _toy(a, 1, n_w=5)
    with pytest.raises(TypeError):
        sv.value_iteration(J0, report_time=False, risk=(0.5, 0.5))
    sv.perturb_proba = [np.array([0.5, 0.6, -0.1, 0.0, 0.0])]
    with pytest.raises(ValueError, match="probabilities"):
        sv.value_iteration(J0, report_time=False, risk=product.MeanCVaR(*RISK))
    sv.perturb_proba = [np.array([0.5, np.nan, 0.5, 0.0, 0.0])]
    with pytest.raises(ValueError, match="probabilities"):
        sv.eval_policy(np.zeros(sv._state_grid_shape + (1,)), 2, report_time=False,
                       risk=product.MeanCVaR(*RISK))


@pytest.mark.parametrize("which", ["A", "B", "AF", "BF", "CF"])
def test_risk_tables(product, which):
    """layout A and CF tables serve both operators; B, AF and BF problems get dense layout-A tables
    under risk, kept beside the expectation's (at most one entry of each kind)"""
    import workloads as wl
    a = _Api(product, "model")
    if which == "CF":
        sv = wl.storage_ar1(a, n_E=40, n_P=3, n_w=3, steps=(2.0, 0.1)).solver
        sv.table_layout, sv.column_hoist = "state_minor", "on"
    else:
        sv = _toy(a, 2) if which in ("A", "B") else \
            __import__("test_parity")._two_perturbations(a, "split")
        sv.table_layout = "state_minor" if which in ("B", "BF") else "control_minor"
        if which in ("A", "B"):
            sv.table_compress = "off"
    settings = (sv.table_layout, sv.table_compress, sv.column_hoist, sv.slab_axis)
    J0 = np.random.default_rng(1).standard_normal(sv._state_grid_shape)
    sv.value_iteration(J0, report_time=False)
    T0 = sv.last_tables
    assert T0.layout_name == LAYOUT[which]
    sv.value_iteration(J0, report_time=False, risk=product.MeanCVaR(*RISK))
    T1 = sv.last_tables
    if which in ("A", "CF"):
        assert T1 is T0 and len(sv._table_cache) == 1
    else:
        assert T1.layout_name == "control_minor" and len(sv._table_cache) == 2
    assert (sv.table_layout, sv.table_compress, sv.column_hoist, sv.slab_axis) == settings
    sv.value_iteration(J0, report_time=False)
    assert sv.last_tables is T0
    sv.value_iteration(J0, report_time=False, risk=product.MeanCVaR(0.3, 0.1))
    assert sv.last_tables is T1
    # a risk sweep alone (nothing cached): CF where it applies, else dense A
    sv.clear_tables()
    sv.value_iteration(J0, report_time=False, risk=product.MeanCVaR(*RISK))
    assert sv.last_tables.layout_name == ("column_factored" if which == "CF" else "control_minor")


def _check_vi(sv, so, J0, risk_pkg):
    J, pol = sv.value_iteration(J0, report_time=False, risk=risk_pkg)
    with np.errstate(invalid="ignore"):
        Jo, polo = so.value_iteration(J0)
    assert np.array_equal(pol, polo)
    assert same(J, Jo)
    return J, pol


@pytest.mark.parametrize("d,n_w", [(1, 5), (2, 9), (3, 13), (4, 16), (2, 1)])
def test_value_iteration_against_port(api, product, d, n_w):
    sv, so = _toy(api, d, n_w=n_w), _toy(rp.port_api(RISK), d, n_w=n_w)
    rng = np.random.default_rng(d)
    J0 = rng.standard_normal(sv._state_grid_shape)
    _check_vi(sv, so, J0, product.MeanCVaR(*RISK))
    # NaN and +-inf nodes of J
    J1 = J0.copy().reshape(-1)
    J1[rng.choice(J1.size, 3, replace=False)] = [np.inf, -np.inf, np.nan]
    _check_vi(sv, so, J1.reshape(J0.shape), product.MeanCVaR(*RISK))
    # relative DP
    Jr = J0 - J0[sv._state_ref_ind]
    (Jd, ref), pol = sv.value_iteration((Jr, 0.0), rel_dp=True, report_time=False, risk=product.MeanCVaR(*RISK))
    (Jdo, refo), polo = so.value_iteration((Jr, 0.0), rel_dp=True)
    assert np.array_equal(pol, polo) and same(Jd, Jdo) and ref == refo


def test_solver_methods_against_port(api, product):
    R = product.MeanCVaR(*RISK)
    sv, so = _toy(api, 2, n_w=9), _toy(rp.port_api(RISK), 2, n_w=9)
    shape = sv._state_grid_shape
    J, pol, info = sv.solve_value_iteration(np.zeros(shape), max_iter=4, risk=R)
    Jo = np.zeros(shape)
    for _ in range(4):
        Jo, polo = so.value_iteration(Jo)
    assert same(J, Jo) and np.array_equal(pol, polo)
    Je = sv.eval_policy(pol, 5, report_time=False, risk=R)
    assert same(Je, so.eval_policy(polo, 5))
    (Jr, ref) = sv.eval_policy(pol, 5, rel_dp=True, report_time=False, risk=R)
    (Jro, refo) = so.eval_policy(polo, 5, rel_dp=True)
    assert same(Jr, Jro) and ref == refo
    Jp, pp = sv.policy_iteration(pol, 3, 2, risk=R)
    Jpo, ppo = so.policy_iteration(polo, 3, 2)
    assert same(Jp, Jpo) and np.array_equal(pp, ppo)


@pytest.mark.parametrize("mode", ["auto", "per_instant"])
def test_bellman_recursion_against_port(api, product, mode):
    sv, so = _timedep(api), _timedep(rp.port_api(RISK))
    sv.recursion_mode = mode
    J_fin = np.random.default_rng(3).standard_normal(sv._state_grid_shape)
    J, pol = sv.bellman_recursion(6, J_fin, report_time=False, risk=product.MeanCVaR(*RISK))
    Jo, polo = so.bellman_recursion(6, J_fin)
    assert same(J, Jo) and np.array_equal(pol, polo)
    if mode == "auto" and api.backend == "model":
        assert sv.last_recursion is not None          # the fast path ran


# ---------------------------------------------------------------------------
# GPU: weight 0, the benchmark configurations, optimality
# ---------------------------------------------------------------------------
def _config(api, which):
    import workloads as wl
    if which == "#1":
        return wl.inventory(api).solver
    if which == "#3":
        return wl.storage_ar1(api).solver
    if which == "#4":
        return wl.searev(api).solver
    if which == "#5-small":
        return wl.storage_ar1_large(api, n_E=200, n_P=50).solver
    if which == "#5":
        return wl.storage_ar1_large(api).solver
    raise KeyError(which)


@gpu
@pytest.mark.parametrize("which", ["#1", "#3", "#5-small", "#5"])
def test_weight_zero_equals_expectation(cuda_api, product, which):
    sv = _config(cuda_api, which)
    J0 = np.random.default_rng(11).standard_normal(sv._state_grid_shape)
    J, pol = sv.value_iteration(J0, report_time=False)
    Jr, polr = sv.value_iteration(J0, report_time=False, risk=product.MeanCVaR(0.9, 0.0))
    assert same(J, Jr) and np.array_equal(pol, polr)
    assert sv.last_tables.layout_name in ("control_minor", "column_factored")
    sv.clear_tables()


@gpu
@pytest.mark.parametrize("which", ["#1", "#3", "#4", "#5"])
def test_risk_sweep_against_port(cuda_api, product, which):
    sv = _config(cuda_api, which)
    so = _config(rp.port_api(RISK), which)
    shape = sv._state_grid_shape
    n = int(np.prod(shape))
    J0 = np.random.default_rng(12).standard_normal(shape)
    J, pol = sv.value_iteration(J0, report_time=False, risk=product.MeanCVaR(*RISK))
    T = sv.last_tables
    states = np.arange(n) if n <= 3000 else np.random.default_rng(13).choice(n, 1000, replace=False)
    Jo, idx = so.value_iteration_states(J0, states)
    assert same(J.reshape(-1)[states], Jo)
    # policies: the argmin maps to the port's control values
    nc = pol.shape[-1]
    for j, s in enumerate(states[:200]):
        ind_x = np.unravel_index(int(s), shape)
        x_k = tuple(g[i] for g, i in zip(so.state_grid, ind_x))
        grids, dims = so.control_grids(x_k)
        ind_u = np.unravel_index(int(idx[j]), dims)
        assert np.array_equal(pol.reshape(-1, nc)[s], [grids[c][ind_u[c]] for c in range(nc)])
    assert T.layout_name == ("column_factored" if which == "#5" else "control_minor")
    sv.clear_tables()


@gpu
def test_value_iteration_equals_solve_on_config5(cuda_api, product):
    R = product.MeanCVaR(*RISK)
    sv = _config(cuda_api, "#5")
    J0 = np.random.default_rng(14).standard_normal(sv._state_grid_shape)
    J, pol = sv.value_iteration(J0, report_time=False, risk=R)
    Js, pols, _ = sv.solve_value_iteration(J0, max_iter=1, risk=R)
    assert same(J, Js) and np.array_equal(pol, pols)
    sv.clear_tables()


def _inside(api):
    """a stationary system whose next states stay on the grid (interpolation weights in [0, 1]:
    the backups are monotone, which optimality and the order in the weight rest on)"""
    import scipy.stats as stats

    def dyn(x0, x1, u, w):
        return (np.clip(0.7 * x0 + 0.4 * u, -1.0, 2.0), np.clip(0.6 * x1 + 0.3 * u * x0 + 0.5 * w, -1.0, 1.5))

    def box(x0, x1):
        return ((-1.0, 1.0),)

    def cost(x0, x1, u, w):
        return x0 ** 2 + 0.5 * x1 ** 2 + 0.1 * u ** 2 + 0.3 * w * u

    sys = api.SysDescription((2, 1, 1), name='inside the grid')
    sys.dyn, sys.control_box, sys.cost = dyn, box, cost
    sys.perturb_laws = [stats.norm(0, 0.4)]
    sv = api.DPSolver(sys)
    sv.discretize_state(-1.0, 2.0, 7, -1.0, 1.5, 6)
    sv.discretize_perturb(-1.0, 1.0, 9)
    sv.control_steps = (2.0 / 20,)
    return sv


@gpu
def test_optimality_and_weight_monotonicity(cuda_api, product):
    sv = _inside(cuda_api)
    shape = sv._state_grid_shape
    n = 6
    _, pol_neutral, _ = sv.solve_value_iteration(np.zeros(shape), max_iter=n)
    prev = None
    for wgt in (0.0, 0.3, 0.7, 1.0):
        R = product.MeanCVaR(0.8, wgt)
        J, _, _ = sv.solve_value_iteration(np.zeros(shape), max_iter=n, risk=R)
        Je = sv.eval_policy(pol_neutral, n, report_time=False, risk=R)
        assert np.all(J <= Je + 1e-12 * np.maximum(np.abs(Je), 1.0))
        if prev is not None:
            assert np.all(J >= prev - 1e-12 * np.maximum(np.abs(prev), 1.0))
        prev = J


@gpu
def test_last_kernel_names(cuda_api, product):
    sv = _toy(cuda_api, 3, n_w=13)
    J0 = np.zeros(sv._state_grid_shape)
    sv.value_iteration(J0, report_time=False, risk=product.MeanCVaR(*RISK))
    assert _cabi.last_kernel() == "k_sweep_risk<3,16>"
    sv.eval_policy(np.zeros(sv._state_grid_shape + (1,)), 2, report_time=False, risk=product.MeanCVaR(*RISK))
    assert _cabi.last_kernel() == "k_policy_eval_risk<3,16,0>"


@gpu
def test_raw_abi_refusals(cuda_api, product):
    import workloads as wl
    sv = wl.storage_ar1(cuda_api, n_E=40, n_P=3, n_w=3, steps=(2.0, 0.1)).solver
    sv.table_layout, sv.column_hoist = "state_minor", "on"
    J0 = np.zeros(sv._state_grid_shape)
    sv.value_iteration(J0, report_time=False)
    T = sv.last_tables
    assert T.layout_name == "column_factored"
    lib = _cabi.load_library()
    eng = sv.engine
    r = product.MeanCVaR(*RISK).c_struct()
    n0 = lib.sdp_launch_count()
    for field, value in (("col_pairs", 1), ("layout", _cabi.LAYOUT_STATE_MINOR_FACTORED),
                         ("layout", _cabi.LAYOUT_STATE_MINOR)):
        bad = _cabi.SdpTables.from_buffer_copy(T.c_tables)
        setattr(bad, field, value)
        rc = lib.sdp_sweep_risk_partials(ctypes.byref(T.grid), ctypes.byref(bad), ctypes.byref(r),
                                         eng._ptr(T.part_val), eng._ptr(T.part_val), eng._ptr(T.part_idx),
                                         eng.stream)
        assert rc == -1
    assert lib.sdp_launch_count() == n0
    sv.value_iteration(J0, report_time=False, risk=product.MeanCVaR(*RISK))
    TA = sv.last_tables
    n1 = lib.sdp_launch_count()
    for bad in ((0.0, 0.0, 1.0, 0.0), (2.0, 0.5, 1.5, 0.0), (2.0, 0.5, 0.5, -0.1), (np.inf, 0.0, 1.0, 0.0)):
        rb = _cabi.SdpRisk(*bad)
        rc = lib.sdp_sweep_risk_partials(ctypes.byref(TA.grid), ctypes.byref(TA.c_tables), ctypes.byref(rb),
                                         eng._ptr(TA.part_val), eng._ptr(TA.part_val), eng._ptr(TA.part_idx),
                                         eng.stream)
        assert rc == -1
    assert lib.sdp_launch_count() == n1
