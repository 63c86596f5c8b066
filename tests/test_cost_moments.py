"""Moments of a policy's total cost: DPSolver.cost_moments (sdp_cost_moments of
include/sdp_b200.h).

For every start state the recursion gives the mean, the variance and the third central moment
of the stage cost accumulated before a target set (or over the whole horizon).  It is checked:
- against a brute-force enumeration of every (node, corner) sequence with its probability, which
  gives the exact law of the cost (inventory n <= 4, a few start states of storage-AR1 n <= 3):
  this checks the derivation, not only the recursion;
- against the exact chain: one table of (x, w, corner) entries per node, built from dyn/cost and
  the oracle's cell search as tests/test_forward.py's `oracle_chain`, the centred sums evaluated
  entry by entry; every step of the history, both clamp settings, with and without a target;
- against identities: first_passage's cost and eval_policy bit for bit, var >= 0 with clamped
  weights, zero spread on a deterministic grid-node system, exact scaling with a doubled cost,
  n = 0, a converged `tol` run equal to the fixed run;
- on the GPU, bit for bit against the numpy model below (the same operations in the same order) on
  the device's own tables, run to run, across launch shapes and split calls; and statistically
  against 10^6 paths of sample_paths on config #5.

CPU suite ("model"): the host code drives the numpy model (CostMomentsFakeLib).  GPU suite
("cuda"): the real library.
"""
import ctypes

import numpy as np
import pytest

from fake_lib import _arr, _grid
from oracle import oracle as oc
from test_first_passage import CASES, FirstPassageFakeLib, _fp_case, _mask_bits, outside_count
from test_forward import RTOL, rel_l1
from test_sample_paths import _z

gpu = pytest.mark.gpu


# ---------------------------------------------------------------------------
# numpy model of sdp_cost_moments
# ---------------------------------------------------------------------------
def model_steps(strides, W, g_per_w, p, C, L, G, tmask, clamp, V, n_steps, hist=None):
    """n_steps steps from V (n, 4) with the tables C (W, n), L (d, W, n), G (W|1, n), p (W,);
    hist (n_steps+1, n, 4) receives every step.  Returns (V after n_steps, sup-norm change of the
    last step)"""
    d, n = L.shape[0], V.shape[0]
    if clamp:
        L = np.where((L < 0.0) | np.isnan(L), 0.0, np.where(L > 1.0, 1.0, L))
    resid = 0.0
    if hist is not None:
        hist[0] = V
    for step in range(n_steps):
        old = V
        with np.errstate(all="ignore"):
            def lerp(base, k, lam, leaf):
                if k == d:
                    return leaf(base)
                a = lerp(base, k + 1, lam, leaf)
                b = lerp(base + strides[k], k + 1, lam, leaf)
                m = 1.0 - lam[k]
                return tuple(m * x + lam[k] * y for x, y in zip(a, b))

            M = np.zeros(n)
            for w in range(W):
                gv = G[w if g_per_w else 0]
                M = M + (gv + lerp(C[w], 0, L[:, w], lambda c: (old[c, 0],))[0]) * p[w]
            Var, K3 = np.zeros(n), np.zeros(n)
            for w in range(W):
                gv = G[w if g_per_w else 0]

                def leaf(c):
                    dl = (gv + old[c, 0]) - M
                    dd = dl * dl
                    return old[c, 1] + dd, old[c, 2] + dl * (3.0 * old[c, 1] + dd)

                a, b = lerp(C[w], 0, L[:, w], leaf)
                Var = Var + a * p[w]
                K3 = K3 + b * p[w]
            new = np.zeros((n, 4))
            new[:, 0] = np.where(tmask, 0.0, M)
            new[:, 1] = np.where(tmask, 0.0, Var)
            new[:, 2] = np.where(tmask, 0.0, K3)
            resid = float(np.max(np.abs(new[:, :3] - old[:, :3])))
        V = new
        if hist is not None:
            hist[step + 1] = V
    return V, resid


class CostMomentsFakeLib(FirstPassageFakeLib):
    """the models of FirstPassageFakeLib plus the model of sdp_cost_moments"""

    def sdp_cost_moments(self, gref, W, g_per_w, p, cell, lam, lam_plane, g, n_states, target, clamp, V_a, V_b,
                         n_steps, hist, resid_out, counters, stream):
        d, _, _, orders = _grid(gref)
        n = int(np.prod(orders))
        assert n_states == n
        strides = [int(np.prod(orders[k + 1:])) for k in range(d)]
        C = _arr(cell, W * n, ctypes.c_int32).astype(np.int64).reshape(W, n)
        L = np.stack([_arr(lam.value + 8 * k * lam_plane, W * n, ctypes.c_double).reshape(W, n)
                      for k in range(d)])
        G = _arr(g, (W if g_per_w else 1) * n, ctypes.c_double).reshape(-1, n)
        tmask = _mask_bits(_arr(target, (n + 31) // 32, ctypes.c_uint32), n) if (target.value or 0) else \
            np.zeros(n, bool)
        A = _arr(V_a, 4 * n, ctypes.c_double).reshape(n, 4)
        B = _arr(V_b, 4 * n, ctypes.c_double).reshape(n, 4)
        H = _arr(hist, (n_steps + 1) * 4 * n, ctypes.c_double).reshape(-1, n, 4) if (hist.value or 0) else None
        V, resid = model_steps(strides, W, g_per_w, _arr(p, W, ctypes.c_double), C, L, G, tmask, clamp,
                               A.copy(), n_steps, H)
        if n_steps:
            (A if n_steps % 2 == 0 else B)[:] = V
            if counters.value or 0:
                _arr(counters, 1, ctypes.c_int64)[0] += outside_count(L, tmask)
        if resid_out.value or 0:
            _arr(resid_out, 1, ctypes.c_double)[0] = resid if n_steps else 0.0
        self.launches += n_steps
        return 0


class _Api(object):
    def __init__(self, pkg, backend):
        self.pkg = pkg
        self.backend = backend
        self.SysDescription = pkg.SysDescription

    def DPSolver(self, sys, **kw):
        if self.backend == "model":
            kw["_test_lib"] = CostMomentsFakeLib()
        return self.pkg.DPSolver(sys, **kw)


@pytest.fixture(scope="module", params=[pytest.param("model", id="model"),
                                        pytest.param("cuda", marks=gpu, id="cuda")])
def api(request, product):
    return _Api(product, request.param)


@pytest.fixture(scope="module")
def cuda_api(product):
    return _Api(product, "cuda")


def _run(solver, pol, n, td, **kw):
    return solver.cost_moments(pol, n_steps=None if td else n, report_time=False, **kw)


def _same_bits(a, b):
    return a.shape == b.shape and np.array_equal(a.view(np.int64), b.view(np.int64))


# ---------------------------------------------------------------------------
# the exact chain: (x, w, corner) entries from dyn/cost and the oracle's cell search
# ---------------------------------------------------------------------------
def node_entries(solver, pol, t_k=None, clamp=False):
    """(p [W], g [W, n], y [2^d, W, n], phi [2^d, W, n]) of the policy `pol` at instant t_k: the
    stage cost of every (x, w) and the next state's cell corners with their weights (clamped to
    [0, 1], NaN: 0, with clamp), as oracle_chain of tests/test_forward.py builds them"""
    sys = solver.sys
    grids = [np.asarray(g, dtype=float) for g in solver.state_grid]
    dims = tuple(len(g) for g in grids)
    n, d = int(np.prod(dims)), len(dims)
    mesh = [m.reshape(n, 1) for m in np.meshgrid(*grids, indexing="ij")]
    u = [pol[..., i].reshape(n, 1) for i in range(pol.shape[-1])]
    if len(solver.perturb_grid):
        ws = np.meshgrid(*[np.asarray(g, dtype=float) for g in solver.perturb_grid], indexing="ij")
        ps = np.meshgrid(*[np.asarray(q, dtype=float) for q in solver.perturb_proba], indexing="ij")
        w_args = tuple(w.reshape(1, -1) for w in ws)
        p = np.prod(ps, axis=0).reshape(-1)
    else:
        w_args, p = (), np.ones(1)
    W = len(p)
    args = ((t_k,) if t_k is not None else ()) + tuple(mesh) + tuple(u) + w_args
    nxt = [np.broadcast_to(np.asarray(c, dtype=float), (n, W)) for c in sys.dyn(*args, **sys.params)]
    g = np.broadcast_to(np.asarray(sys.cost(*args, **sys.params), dtype=float), (n, W)).T
    S = np.stack([c.T.reshape(-1) for c in nxt])           # [d][W*n], w-major
    cell, lam = oc.cell_search([a[0] for a in grids], [a[-1] for a in grids], np.array(dims), S)
    if clamp:
        lam = np.clip(np.nan_to_num(lam, nan=0.0), 0.0, 1.0)
    strides = [int(np.prod(dims[k + 1:])) for k in range(d)]
    ys, phis = [], []
    for eps in range(1 << d):
        y = cell.astype(np.int64)
        c = np.ones(W * n)
        for k in range(d):
            bit = (eps >> k) & 1
            y = y + bit * strides[k]
            c = c * (lam[k] if bit else 1 - lam[k])
        ys.append(y.reshape(W, n))
        phis.append(c.reshape(W, n))
    return p, np.ascontiguousarray(g), np.stack(ys), np.stack(phis)


def oracle_moments(solver, pol, target, n_steps, clamp, td):
    """[(M_k, V_k, K_k) for k = 0 .. n] of the exact chain, the centred sums taken entry by entry:
    V = sum p_w phi (V(y) + d^2), K = sum p_w phi (K(y) + 3 V(y) d + d^3), d = g + M(y) - m"""
    N = int(np.prod(solver._state_grid_shape))
    t = np.zeros(N, bool) if target is None else target.reshape(-1)
    M, V, K = np.zeros(N), np.zeros(N), np.zeros(N)
    out = [(M, V, K)]
    fixed = None if td else node_entries(solver, pol, clamp=clamp)
    for k in range(n_steps - 1, -1, -1):
        p, g, y, phi = node_entries(solver, pol[k], t_k=k, clamp=clamp) if td else fixed
        q = p[None, :, None] * phi                             # [corner, w, x]
        gy = g[None] + M[y]
        m = (q * gy).sum(axis=(0, 1))
        dl = gy - m
        Vn = (q * (V[y] + dl ** 2)).sum(axis=(0, 1))
        Kn = (q * (K[y] + 3.0 * V[y] * dl + dl ** 3)).sum(axis=(0, 1))
        M, V, K = np.where(t, 0.0, m), np.where(t, 0.0, Vn), np.where(t, 0.0, Kn)
        out.append((M, V, K))
    return out[::-1]


@pytest.mark.parametrize("with_target", [True, False], ids=["target", "notarget"])
@pytest.mark.parametrize("clamp", [True, False], ids=["clamp", "noclamp"])
@pytest.mark.parametrize("which", CASES)
def test_against_the_exact_chain(api, which, clamp, with_target):
    solver, pol, n, td, target = _fp_case(api, which)
    target = target if with_target else None
    dims = solver._state_grid_shape
    mean, var, third, info = _run(solver, pol, n, td, target=target, clamp=clamp, history=True)
    assert mean.shape == var.shape == third.shape == (n + 1,) + dims
    assert info["n_steps"] == n and not info["converged"] and info["residuals"] == []
    ref = oracle_moments(solver, pol, target, n, clamp, td)
    # Where the spread is zero (a cost that does not depend on w, one step left), V and K are the
    # rounding noise of the deviations d = g + M(y) - m, whose absolute error is a few ulp of the
    # largest mean s; rel_l1 of noise against noise means nothing.  So V and K also get the
    # absolute floor that an error e = 1e-13 s in every d makes, per state: 2 e sqrt(V) + e^2 in
    # d^2, and 3 e (V + d^2) + e^2 (...) in 3 V d + d^3.
    N = mean[0].size
    e = 1e-13 * float(np.abs(mean).max())
    vmax = float(np.abs(var).max())
    floor = {"M": 0.0, "V": N * (2.0 * e * np.sqrt(vmax) + e * e), "K": N * (6.0 * e * vmax + e * e)}
    for k in range(n + 1):
        for got, want, name in zip((mean[k], var[k], third[k]), ref[k], "MVK"):
            err = float(np.abs(got.reshape(-1) - want).sum())
            assert err <= RTOL * float(np.abs(want).sum()) + floor[name], \
                (which, clamp, k, name, rel_l1(got, want), err, floor[name])
    # without history: the values of step 0, bit for bit
    m0, v0, k0, info0 = _run(solver, pol, n, td, target=target, clamp=clamp)
    for a, b in ((m0, mean[0]), (v0, var[0]), (k0, third[0])):
        assert _same_bits(a, b)
    assert info0["outside_share"] == info["outside_share"] and 0.0 <= info["outside_share"] <= 1.0
    print(which, "clamp" if clamp else "noclamp", "target" if with_target else "no target",
          "std range", float(np.sqrt(np.maximum(var[0], 0)).min()), float(np.sqrt(np.maximum(var[0], 0)).max()))


# ---------------------------------------------------------------------------
# brute force: the exact law of the cost, every (node, corner) sequence enumerated
# ---------------------------------------------------------------------------
def brute_force_law(solver, pol, target, n_steps, clamp, starts):
    """(start index, cost, probability) of every sequence of (node, corner) choices from the start
    states `starts` (flat indices) over n_steps steps; the cost stops at the first step in
    `target`.  With clamp=False the weights, and so the probabilities, may be negative"""
    p, g, y, phi = node_entries(solver, pol, clamp=clamp)
    t = np.zeros(y.shape[-1], bool) if target is None else target.reshape(-1)
    C, W = y.shape[0], len(p)
    src = np.asarray(starts, dtype=np.int64)
    state, cost, prob = src.copy(), np.zeros(len(src)), np.ones(len(src))
    alive = np.ones(len(src), bool)
    for _ in range(n_steps):
        alive &= ~t[state]
        a = np.flatnonzero(alive)
        s = state[a]
        # children of every live sequence, node-major then corner
        ny = y[:, :, s].transpose(2, 1, 0).reshape(-1)                          # [seq, w, corner]
        nq = (prob[a][:, None, None] * p[None, :, None] * phi[:, :, s].transpose(2, 1, 0)).reshape(-1)
        nc = np.repeat((cost[a][:, None] + g[:, s].T).reshape(-1), C)
        keep = ~alive
        src = np.concatenate([src[keep], np.repeat(src[a], W * C)])
        state = np.concatenate([state[keep], ny])
        cost = np.concatenate([cost[keep], nc])
        prob = np.concatenate([prob[keep], nq])
        alive = np.concatenate([alive[keep], np.ones(ny.size, bool)])
    return src, cost, prob


@pytest.mark.parametrize("clamp", [True, False], ids=["clamp", "noclamp"])
@pytest.mark.parametrize("which", ["inventory", "storage_ar1"])
def test_against_the_brute_force_law(api, which, clamp):
    """the mean, variance and third central moment of the enumerated law, within 1e-10 of the
    scale of each sum (the sum of |q| |G - mean|^j: the law's terms cancel, the recursion's do not
    in the same way)"""
    solver, pol, _, _, target = _fp_case(api, which)
    dims = solver._state_grid_shape
    N = int(np.prod(dims))
    if which == "inventory":                           # d = 1, W = 4: every state, n <= 4
        starts, horizons = np.arange(N), range(1, 5)
    else:                                              # d = 2, W = 9: (36)^n sequences per start
        starts, horizons = np.array([0, 5 * dims[1] + 3, 20 * dims[1] + 30, N // 2 + 7, N - 1]), range(1, 4)
    for n in horizons:
        for tgt in (target, None):
            mean, var, third, _ = solver.cost_moments(pol, n, target=tgt, clamp=clamp, report_time=False)
            src, G, q = brute_force_law(solver, pol, tgt, n, clamp, starts)
            for j, x in enumerate(starts):
                sel = src == x
                qx, Gx = q[sel], G[sel]
                assert abs(qx.sum() - 1.0) <= 1e-12
                mu = float((qx * Gx).sum())
                dv = Gx - mu
                want = (mu, float((qx * dv ** 2).sum()), float((qx * dv ** 3).sum()))
                scale = [float((np.abs(qx) * np.abs(f)).sum()) for f in (Gx, dv ** 2, dv ** 3)]
                # and, where the spread is zero, the rounding noise of the recursion's deviations
                # (absolute error e, as in test_against_the_exact_chain)
                e = 1e-13 * float(np.abs(Gx).max())
                floor = (0.0, 2.0 * e * np.sqrt(abs(want[1])) + e * e, 6.0 * e * abs(want[1]) + e * e)
                got = (mean.reshape(-1)[x], var.reshape(-1)[x], third.reshape(-1)[x])
                for name, a, b, s, f in zip("MVK", got, want, scale, floor):
                    assert abs(a - b) <= 1e-10 * s + f, (which, clamp, n, tgt is None, x, name, a, b, s, f)
        print(which, "clamp" if clamp else "noclamp", "n", n, "sequences", G.size)


# ---------------------------------------------------------------------------
# identities
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("which", ["inventory", "storage_ar1", "product-3x2", "pv_storage"])
def test_identities(api, which):
    solver, pol, n, td, target = _fp_case(api, which)
    for clamp in (True, False):
        for tgt in (target, None):
            mean, var, third, info = _run(solver, pol, n, td, target=tgt, clamp=clamp, history=True)
            # the mean is first_passage's cost, bit for bit
            fp_target = np.zeros(target.shape, bool) if tgt is None else tgt
            _, _, cost, fp_info = solver.first_passage(pol, fp_target, None if td else n, clamp=clamp,
                                                       history=True, report_time=False)
            assert _same_bits(mean, cost), (which, clamp, tgt is None)
            assert info["outside_share"] == fp_info["outside_share"]
            if clamp:
                assert np.all(var >= 0.0), float(var.min())
            if tgt is not None:                             # target states: (0, 0, 0) at every step
                assert np.all(mean[:, tgt] == 0.0) and np.all(var[:, tgt] == 0.0) and np.all(third[:, tgt] == 0.0)
    if not td:
        # no target, weights as they are: the mean is eval_policy's, bit for bit
        mean, _, _, _ = solver.cost_moments(pol, n, clamp=False, report_time=False)
        J = solver.eval_policy(pol, n, report_time=False)
        assert _same_bits(mean, J)
        # no step: zeros
        for tgt in (target, None):
            mean, var, third, info = solver.cost_moments(pol, 0, target=tgt, report_time=False)
            assert np.all(mean == 0) and np.all(var == 0) and np.all(third == 0)
            assert info["n_steps"] == 0 and info["outside_share"] == 0.0


def _grid_node_system(api):
    """deterministic, stationary: x in {0, .., 9}, u in {-2, .., 2}, next state x + u, a grid node
    (or, out of the grid, projected onto its boundary node by the clamp)"""
    sys = api.SysDescription((1, 1, 0), name="grid nodes")
    sys.dyn = lambda x, u: (x + u,)
    sys.control_box = lambda x: ((-2, 2),)
    sys.cost = lambda x, u: (x - 4.0) ** 2 + 0.3 * u
    solver = api.DPSolver(sys)
    solver.discretize_state(0, 9, 10)
    solver.control_steps = (1,)
    x = np.arange(10.0)
    pol = np.where(x < 4, 2.0, np.where(x > 6, -1.0, 1.0)).reshape(10, 1)
    return solver, pol


def test_deterministic_grid_nodes_have_no_spread(api):
    solver, pol = _grid_node_system(api)
    target = np.zeros(10, bool)
    target[9] = True
    for tgt in (None, target):
        mean, var, third, _ = solver.cost_moments(pol, 15, target=tgt, history=True, report_time=False)
        assert np.all(var == 0.0) and np.all(third == 0.0)
        assert mean[0].max() > 0.0


def test_doubling_the_cost(api):
    """2g gives exactly (2M, 4V, 8K): every operation scales by a power of two"""
    import workloads as wl
    solver, pol, n, _, target = _fp_case(api, "inventory")
    prob = wl.inventory(api)
    op = prob.sys.cost
    prob.sys.cost = lambda x, u, w: 2.0 * op(x, u, w)
    for clamp in (True, False):
        for tgt in (target, None):
            a = solver.cost_moments(pol, n, target=tgt, clamp=clamp, history=True, report_time=False)
            b = prob.solver.cost_moments(pol, n, target=tgt, clamp=clamp, history=True, report_time=False)
            for f, x, y in zip((2.0, 4.0, 8.0), a[:3], b[:3]):
                assert _same_bits(f * x, y), (clamp, tgt is None, f)
            assert np.any(a[2] != 0.0)


def test_tol_run_equals_the_fixed_run(api):
    """inventory, target the three lowest stock levels, reached almost surely from everywhere: a
    converged tol run is the fixed run of the same length bit for bit"""
    solver, pol, _, _, _ = _fp_case(api, "inventory")
    target = np.zeros(solver._state_grid_shape, dtype=bool)
    target[:3] = True
    mean, var, third, info = solver.cost_moments(pol, 20000, target=target, tol=1e-9, check_every=25,
                                                 report_time=False)
    m = info["n_steps"]
    assert info["converged"] and m % 25 == 0 and len(info["residuals"]) == m // 25 and m < 20000
    assert info["residuals"][-1] <= 1e-9 < info["residuals"][-2]
    m2, v2, k2, info2 = solver.cost_moments(pol, m, target=target, report_time=False)
    for a, b in ((mean, m2), (var, v2), (third, k2)):
        assert _same_bits(a, b)
    assert info2["outside_share"] == info["outside_share"]
    # the mean is first_passage's converged cost
    _, _, cost, _ = solver.first_passage(pol, target, m, report_time=False)
    assert _same_bits(mean, cost)
    hist, _, _, info3 = solver.cost_moments(pol, 20000, target=target, tol=1e-9, check_every=25, history=True,
                                            report_time=False)
    assert info3["n_steps"] == m and hist.shape == (m + 1,) + mean.shape
    assert _same_bits(hist[0], mean) and np.all(hist[m] == 0.0)
    print("inventory: converged after", m, "steps; std of the cost before tau in",
          float(np.sqrt(var).min()), float(np.sqrt(var).max()))


def test_argument_checks(api):
    solver, pol, n, _, target = _fp_case(api, "storage_ar1")

    def run(**kw):
        args = dict(pol=pol, n_steps=3, target=target, report_time=False)
        args.update(kw)
        return solver.cost_moments(**args)

    with pytest.raises(ValueError, match=r"array `pol` should be of shape"):
        run(pol=pol[..., :1])
    with pytest.raises(ValueError, match=r"array `target` should be of shape"):
        run(target=target[:-1])
    with pytest.raises(ValueError, match=r"array `target` should be of shape"):
        run(target=target.T)
    with pytest.raises(ValueError, match=r"boolean"):
        run(target=target.astype(int))
    with pytest.raises(ValueError, match=r"boolean"):
        run(target=target.astype(float))
    with pytest.raises(ValueError, match=r"n_steps"):
        run(n_steps=-1)
    with pytest.raises(ValueError, match=r"n_steps is required"):
        run(n_steps=None)
    for c in (0, -2):
        with pytest.raises(ValueError, match=r"check_every"):
            run(check_every=c, tol=1e-9)
    with pytest.raises(ValueError, match=r"tol needs a target"):
        run(target=None, tol=1e-9)
    # time-dependent system
    tsolver, tpol, _, _, ttarget = _fp_case(api, "pv_storage")
    with pytest.raises(ValueError, match=r"array `pol` should be of shape"):
        tsolver.cost_moments(tpol[0], report_time=False)
    with pytest.raises(ValueError, match="exceeds"):
        tsolver.cost_moments(tpol[:10], n_steps=11, report_time=False)
    with pytest.raises(ValueError, match="tol needs a stationary system"):
        tsolver.cost_moments(tpol, target=ttarget, tol=1e-9, report_time=False)


# ---------------------------------------------------------------------------
# GPU: bit identity with the model, determinism, config #5 against sample_paths
# ---------------------------------------------------------------------------
def _model_on_device_tables(solver, pol, target, n, td, clamp):
    """the model, instant by instant on the device's own tables (read back): the history in the
    order of cost_moments (entry k = step k) and the outside share"""
    eng = solver.engine
    dims = solver._state_grid_shape
    N = int(np.prod(dims))
    tmask = np.zeros(N, bool) if target is None else target.reshape(-1)
    V = np.zeros((N, 4))
    hist = [V]
    count = entries = 0
    for k in (range(n - 1, -1, -1) if td else [None]):
        P = eng.build_policy_tables(solver, np.asarray(pol[k] if td else pol, dtype=float), t_k=k,
                                    deterministic=True)
        d, W = P.grid.d, P.W
        strides = [int(np.prod(dims[j + 1:])) for j in range(d)]
        C = P.cell.cpu().numpy()[:W * N].astype(np.int64).reshape(W, N)
        L = P.lam.cpu().numpy()[:d * P.lam_plane].reshape(d, W, N)
        G = P.g.cpu().numpy().reshape(-1, N)
        steps = 1 if td else n
        H = np.zeros((steps + 1, N, 4))
        V, _ = model_steps(strides, W, P.g_per_w, P.p.cpu().numpy(), C, L, G, tmask, clamp, V, steps, H)
        hist.extend(H[1:])
        if steps:
            count += outside_count(L, tmask)
            entries += W * N
    H = np.stack(hist[::-1])
    return H, count / entries if entries else 0.0


@gpu
@pytest.mark.parametrize("with_target", [True, False], ids=["target", "notarget"])
@pytest.mark.parametrize("clamp", [True, False], ids=["clamp", "noclamp"])
@pytest.mark.parametrize("which", CASES)
def test_kernel_bit_identical_to_the_model(cuda_api, which, clamp, with_target):
    from stodynprog_b200 import _cabi
    solver, pol, n, td, target = _fp_case(cuda_api, which)
    target = target if with_target else None
    mean, var, third, info = _run(solver, pol, n, td, target=target, clamp=clamp, history=True)
    assert _cabi.last_kernel().startswith("k_cost_moments<D=%d,%s>" % (len(solver._state_grid_shape),
                                                                        "clamp" if clamp else "noclamp"))
    H, share = _model_on_device_tables(solver, pol, target, n, td, clamp)
    for j, got in enumerate((mean, var, third)):
        want = H[..., j].reshape(got.shape)
        assert _same_bits(got, want), (which, clamp, with_target, "MVK"[j])
    assert info["outside_share"] == share
    print(which, "clamp" if clamp else "noclamp", "target" if with_target else "no target", "outside share", share)


def _device_setup(solver, pol, target):
    eng = solver.engine
    P = eng.build_policy_tables(solver, np.asarray(pol, dtype=float), deterministic=True)
    mask = eng.to_device(solver._target_mask(target)) if target is not None else None
    return eng, P, mask


@gpu
@pytest.mark.parametrize("with_target", [True, False], ids=["target", "notarget"])
def test_runs_launch_shapes_and_split_calls(cuda_api, with_target):
    import torch
    from stodynprog_b200 import _cabi
    solver, pol, _, _, target = _fp_case(cuda_api, "storage_ar1")
    eng, P, mask = _device_setup(solver, pol, target if with_target else None)
    lib = eng.lib
    N = P.n_states
    n = 41

    def run(threads, split, clamp=True):
        lib.sdp_set_option(b"fp_threads", threads)
        a = torch.zeros(4 * N, dtype=torch.float64, device=eng.device)
        b = torch.empty_like(a)
        cnt = torch.zeros(1, dtype=torch.int64, device=eng.device)
        res = torch.zeros(1, dtype=torch.float64, device=eng.device)
        hist = torch.empty((n + 1) * N * 4, dtype=torch.float64, device=eng.device)
        done = 0
        for k in split:
            out = eng.cost_moments(P, mask, clamp, a, b, k, hist=hist[done * N * 4:(done + k + 1) * N * 4],
                                   resid_out=res, counters=cnt)
            if out is b:
                a, b = b, a
            done += k
        name = _cabi.last_kernel()
        return [t.cpu().numpy() for t in (a.view(torch.int64), hist.view(torch.int64), res.view(torch.int64))], \
            int(cnt.cpu().numpy()[0]) // len(split), name

    try:
        ref, cnt, name = run(0, [n])
        assert name == "k_cost_moments<D=2,clamp>, 256 threads", name
        res = ref[2].view(np.float64)[0]
        vals = ref[0].view(np.float64).reshape(N, 4)
        assert res > 0.0 and vals[:, 3].max() == 0.0 and vals[:, 1].max() > 0.0 and cnt > 0
        for threads, split in [(0, [n]), (96, [n]), (1024, [n]), (0, [17, 24]), (160, [1, 20, 20])]:
            got, c, name = run(threads, split)
            assert str(threads or 256) in name
            assert c == cnt, (threads, split)
            for a, b in zip(ref, got):
                assert np.array_equal(a, b), (threads, split)
    finally:
        lib.sdp_set_option(b"fp_threads", 0)


@gpu
def test_raw_abi_refusals_launch_nothing(cuda_api):
    import torch
    solver, pol, _, _, target = _fp_case(cuda_api, "inventory")
    eng, P, mask = _device_setup(solver, pol, target)
    lib = eng.lib
    N = P.n_states
    a = torch.zeros(4 * N + 2, dtype=torch.float64, device=eng.device)
    b = torch.zeros(4 * N + 2, dtype=torch.float64, device=eng.device)
    ptr = eng._ptr
    null = ctypes.c_void_p(0)

    def call(W=P.W, n_states=P.n_states, lam_plane=P.lam_plane, n_steps=3, p=None, cell=None, V_a=None,
             V_b=None, hist=null):
        return lib.sdp_cost_moments(ctypes.byref(P.grid), W, P.g_per_w, p if p is not None else ptr(P.p),
                                    cell if cell is not None else ptr(P.cell), ptr(P.lam), lam_plane, ptr(P.g),
                                    n_states, ptr(mask), 1, V_a if V_a is not None else ptr(a),
                                    V_b if V_b is not None else ptr(b), n_steps, hist, null, null, eng.stream)

    misaligned = ctypes.c_void_p(a.data_ptr() + 8)
    refusals = {"W = 0": dict(W=0), "n_states": dict(n_states=N - 1), "lam_plane": dict(lam_plane=P.W * N - 1),
                "n_steps < 0": dict(n_steps=-1), "NULL p": dict(p=null), "NULL cell": dict(cell=null),
                "NULL V_a": dict(V_a=null), "NULL V_b": dict(V_b=null), "V_a misaligned": dict(V_a=misaligned),
                "hist misaligned": dict(hist=misaligned)}
    for name, kw in refusals.items():
        before = lib.sdp_launch_count()
        assert call(**kw) == -1, name                      # SDP_EINVAL
        assert b"sdp_cost_moments" in lib.sdp_last_error(), name
        assert lib.sdp_launch_count() == before, name
    before = lib.sdp_launch_count()
    assert call() == 0 and lib.sdp_launch_count() == before + 3


@gpu
def test_nan_makes_the_residual_nan(cuda_api):
    """a NaN value at a corner reaches the residual: a tol run never reports convergence on it"""
    import torch
    solver, pol, _, _, target = _fp_case(cuda_api, "inventory")
    eng, P, mask = _device_setup(solver, pol, target)
    N = P.n_states
    V0 = np.zeros((N, 4))
    V0[N // 2, 2] = np.nan
    a = eng.to_device(V0.reshape(-1))
    b = torch.empty_like(a)
    res = torch.zeros(1, dtype=torch.float64, device=eng.device)
    eng.cost_moments(P, mask, True, a, b, 3, resid_out=res)
    assert np.isnan(res.cpu().numpy()[0])


def _central(x, j):
    return float(((x - x.mean()) ** j).mean())


@gpu
def test_config5_against_sample_paths(cuda_api):
    """config #5 (2000 x 500, W = 9), no target, 20 steps: the sample mean, variance and third
    central moment of the total cost of 10^6 sampled paths against the maps, within 5 standard
    errors estimated from the sample's higher moments (Bonferroni over the six checks), from one
    multi-index and from a start distribution (the maps composed with the formulas of the
    docstring)"""
    import workloads as wl
    prob_ = wl.storage_ar1_large(cuda_api)
    solver = prob_.solver
    _, pol = solver.value_iteration(prob_.J0, report_time=False)
    dims = solver._state_grid_shape
    n, M, K = 20, 1000000, 6
    mean, var, third, info = solver.cost_moments(pol, n, report_time=False)
    assert np.all(var >= 0.0)
    start = (dims[0] // 2, dims[1] // 2)
    mu0 = np.zeros(dims)
    mu0[dims[0] // 4:3 * dims[0] // 4, dims[1] // 4:3 * dims[1] // 4] = 1.0
    mu0 *= np.random.default_rng(5).random(dims)
    w = mu0 / mu0.sum()
    mbar = float((w * mean).sum())
    dev = mean - mbar
    composed = (mbar, float((w * (var + dev ** 2)).sum()), float((w * (third + 3.0 * var * dev + dev ** 3)).sum()))
    print("config #5: outside share", info["outside_share"])
    for start_, want, seed in ((start, (float(mean[start]), float(var[start]), float(third[start])), 41),
                               (mu0, composed, 42)):
        total, _ = solver.sample_paths(pol, start_, n, M, seed=seed, report_time=False)
        m2, m3, m4, m6 = (_central(total, j) for j in (2, 3, 4, 6))
        got = (float(total.mean()), m2 * M / (M - 1), m3)
        se = (np.sqrt(m2 / M), np.sqrt((m4 - m2 ** 2) / M), np.sqrt((m6 - m3 ** 2 - 6.0 * m4 * m2 + 9.0 * m2 ** 3) / M))
        print("start", "index" if isinstance(start_, tuple) else "distribution", "maps", want, "sampled", got,
              "se", se)
        for name, g_, w_, s in zip(("mean", "var", "third"), got, want, se):
            assert abs(g_ - w_) <= _z(K) * s, (name, g_, w_, s)
