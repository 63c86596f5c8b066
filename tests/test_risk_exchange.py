"""Risk sweeps and risk policy evaluation over the peer exchange, N ranks emulated on one GPU
(the harness and hang-free discipline of tests/test_peer_exchange.py: every rank has its own
guarded J, argmin, flag and epoch buffers; the host checks that the flags a wait reads are
published before the wait is enqueued).

- shards of rows (layout A) and of columns (layout CF): every rank runs sdp_sweep_risk_partials on
  its own copy of J, then the fused combine (sdp_sweep_finalize_p2p[_cols]) into every rank's
  buffers; J and the argmin of every rank equal the one-rank risk sweep of the whole grid bit for
  bit, which equals the numpy twin (oracle/risk_port.py);
- sdp_policy_eval_risk_p2p with and without relative DP over 2, 3 and 5 ranks against
  sdp_policy_eval_risk on the whole grid, bit for bit, for d = 1..4 and W = 5, 13.
"""
import ctypes

import numpy as np
import pytest

from oracle import risk_port as rp
from test_parity import _same_bits, _toy
from test_peer_exchange import (LAYOUT_NAMES, SENT_J, Ranks, _case, _col_cuts, _maker, _np, _ptr, _row_cuts,
                                _shards)

pytestmark = pytest.mark.gpu
RISK = (0.8, 0.5)


def _risk(product):
    return product.MeanCVaR(*RISK).c_struct()


def _full_risk_sweep(sv, J0, risk):
    """one single-rank risk sweep of the whole grid through the raw ABI: (J, argmin) in grid order"""
    import torch
    from stodynprog_b200 import _cabi
    eng, T = sv.engine, sv.sweep_tables()
    n = int(np.prod(sv._state_grid_shape))
    Jp = eng.to_device(np.ascontiguousarray(J0, dtype=np.float64).reshape(-1))
    Jo = torch.empty_like(Jp)
    A = torch.empty(n, dtype=torch.int32, device=eng.device)
    _cabi.check(eng.lib.sdp_sweep_risk_partials(ctypes.byref(T.grid), ctypes.byref(T.c_tables), ctypes.byref(risk),
                                                _ptr(Jp), _ptr(T.part_val), _ptr(T.part_idx), eng.stream),
                "sdp_sweep_risk_partials")
    _cabi.check(eng.lib.sdp_sweep_finalize(ctypes.byref(T.c_tables), _ptr(T.part_val), _ptr(T.part_idx),
                                           _ptr(Jo), _ptr(A), eng.stream), "sdp_sweep_finalize")
    return _np(Jo), _np(A)


def _risk_exchange(em, shards, risk, glob_cols=None, cuts=None):
    """one risk sweep of every rank in rank order: partials from its own J[0], fused combine into J[1]"""
    from stodynprog_b200 import _cabi
    lib = em.eng.lib
    for r, (sv, T) in enumerate(shards):
        _cabi.check(lib.sdp_sweep_risk_partials(ctypes.byref(T.grid), ctypes.byref(T.c_tables), ctypes.byref(risk),
                                                _ptr(em.J[r][0]), _ptr(T.part_val), _ptr(T.part_idx), em.eng.stream),
                    "sdp_sweep_risk_partials")
        P = ctypes.byref(em.peers[r][1, True])
        if glob_cols is not None:
            rc = lib.sdp_sweep_finalize_p2p_cols(ctypes.byref(T.c_tables), _ptr(T.part_val), _ptr(T.part_idx),
                                                 _ptr(T.argmin), P, glob_cols, cuts[r], em.eng.stream)
        else:
            rc = lib.sdp_sweep_finalize_p2p(ctypes.byref(T.c_tables), _ptr(T.part_val), _ptr(T.part_idx),
                                            _ptr(T.argmin), P, T.state_begin, em.eng.stream)
        _cabi.check(rc, "sdp_sweep_finalize_p2p")
        em.published(r)
    em.wait_all()
    em.sync()


def _versus_twin(which, sv, J0, J_want, A_want):
    so = _case(rp.port_api(RISK), which)
    n = J_want.size
    states = np.arange(n) if n <= 3000 else np.random.default_rng(3).choice(n, 600, replace=False)
    Jo, idx = so.value_iteration_states(J0, states)
    assert _same_bits(J_want[states], Jo)
    assert np.array_equal(A_want[states], idx)


@pytest.mark.parametrize("layout,axis,which", [("A", "rows", "storage_ar1"), ("CF", "rows", "ar1_w9"),
                                               ("CF", "columns", "ar1_70x70_w9"), ("CF", "columns", "ar1_70x70_w3")])
def test_risk_sweep_shards(product, monkeypatch, layout, axis, which):
    from stodynprog_b200.engine import Engine
    monkeypatch.setattr(Engine, "COLUMN_BANDS", "1")
    risk = _risk(product)
    make = _maker(product, "cuda", layout, which)
    full = make()
    T_full = full.sweep_tables()
    assert T_full.layout_name == LAYOUT_NAMES[layout]
    shape = full._state_grid_shape
    n_grid, n_rows, n_cols = int(np.prod(shape)), shape[0], int(np.prod(shape[1:]))
    J0 = np.random.default_rng(23).standard_normal(shape)
    J_want, A_want = _full_risk_sweep(full, J0, risk)
    _versus_twin(which, full, J0, J_want, A_want)
    for N in (1, 2, 3, 8):
        if axis == "rows":
            cuts = _row_cuts(T_full, N, n_cols, layout == "CF")
        else:
            if N > n_cols:
                continue
            cuts = _col_cuts(T_full, N, n_rows, n_cols)
        shards = _shards(make, cuts, axis)
        em = Ranks(full.engine, N, n_grid)
        em.load(0, J0)
        em.fill(1)
        _risk_exchange(em, shards, risk, glob_cols=n_cols if axis == "columns" else None, cuts=cuts)
        for r in range(N):
            assert _same_bits(_np(em.J[r][1]), J_want), (layout, axis, N, "J of rank", r)
            assert np.array_equal(_np(em.A[r]), A_want), (layout, axis, N, "A[] of rank", r)


def _policy_risk_exchange(sv, pol, cuts, rel, n_iter, risk, J_start):
    """test_peer_exchange._policy_exchange with the risk backups"""
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
    J_start = np.ascontiguousarray(J_start, dtype=np.float64).reshape(-1)
    Ja, Jb = eng.to_device(J_start.copy()), torch.empty(n, dtype=torch.float64, device=eng.device)
    hist = torch.zeros(n_iter, dtype=torch.float64, device=eng.device)
    _cabi.check(eng.lib.sdp_policy_eval_risk(ctypes.byref(P.grid), W, gpw, _ptr(P.p), _ptr(P.cell), _ptr(P.lam),
                                             P.lam_plane, _ptr(P.g), n, 0, n, _ptr(Ja), _ptr(Jb), n_iter, int(rel),
                                             ref, _ptr(hist) if rel else None, ctypes.byref(risk), eng.stream),
                "sdp_policy_eval_risk")
    J_want, h_want = _np(Ja if n_iter % 2 == 0 else Jb), _np(hist)
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
            rc = eng.lib.sdp_policy_eval_risk_p2p(
                ctypes.byref(P.grid), W, gpw, _ptr(P.p), _ptr(x["cell"]), _ptr(x["lam"]), W * x["n"], _ptr(x["g"]),
                x["n"], x["a"], n, _ptr(em.J[r][k_in]), ctypes.byref(em.peers[r][k_out, False]),
                _ptr(x["rc"]) if rel else null, _ptr(x["rl"]) if rel else null, _ptr(x["rg"]) if rel else null,
                ctypes.c_void_p(x["hist"].data_ptr() + 8 * it) if rel else null, ctypes.byref(risk), eng.stream)
            _cabi.check(rc, "sdp_policy_eval_risk_p2p")
            em.published(r)
        em.wait_all()
    em.sync()
    for r, x in enumerate(ranks):
        assert _same_bits(_np(em.J[r][n_iter % 2]), J_want), ("policy J of rank", r, cuts, rel)
        if rel:
            assert _same_bits(_np(x["hist"]), h_want), ("J_ref_out of rank", r)
    return J_want, h_want


@pytest.mark.parametrize("d,n_w", [(1, 5), (2, 13), (3, 5), (4, 13)])
def test_policy_eval_risk_exchange(product, d, n_w):
    from test_risk import _Api
    api = _Api(product, "cuda")
    sv, so = _toy(api, d, "w", n_w=n_w), _toy(rp.port_api(RISK), d, "w", n_w=n_w)
    shape = sv._state_grid_shape
    n = int(np.prod(shape))
    pol = sv.value_iteration(np.random.default_rng(d).standard_normal(shape), report_time=False,
                             risk=product.MeanCVaR(*RISK))[1]
    J_start = np.random.default_rng(40 + d).standard_normal(shape)
    for N in (2, 3, 5):
        cuts = [n * r // N for r in range(N + 1)]
        for rel in (False, True):
            J, h = _policy_risk_exchange(sv, pol, cuts, rel, 5, _risk(product), J_start)
            if N == 2:
                out = so.eval_policy(pol, 5, rel_dp=rel, J_zero=J_start.copy())
                if rel:
                    assert _same_bits(J, out[0].reshape(-1)) and h[-1] == out[1]
                else:
                    assert _same_bits(J, out.reshape(-1))
