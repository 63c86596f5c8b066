"""Distribution propagation under a fixed policy: DPSolver.propagate_distribution and
DPSolver.stationary_distribution (the forward operator mu <- P^T mu of include/sdp_b200.h).

The oracle builds the interpolated Markov chain P as a scipy.sparse matrix, independently of
the product: dyn/cost evaluated here on the policy's grid, next states through the oracle's cell
search, one entry per (state, perturbation node, cell corner).  The product is checked against
`P.T @ mu` iterated, and against eval_policy / bellman_recursion by duality:
<mu_0, J_n> = sum_k c_k, the forward and backward evaluations of the same cost.

CPU suite ("model"): the host code drives a numpy model of the three new entry points (a
subclass of tests/fake_lib.FakeLib).  GPU suite ("cuda"): the real library.
"""
import ctypes

import numpy as np
import pytest
import scipy.sparse as sp

from conftest import golden
from fake_lib import FakeLib, _arr, _grid
from oracle import oracle as oc
from stodynprog_b200 import _cabi

gpu = pytest.mark.gpu
RTOL = 1e-12


class ForwardFakeLib(FakeLib):
    """numpy model of sdp_forward_sizes / _build / _steps: same buffers, same layout (rows by
    destination, entries by source key, pieces of the long rows)"""

    def sdp_forward_sizes(self, d, W, n, nnz, max_pieces, build_b, step_d):
        z = n * W << d
        nnz._obj.value = z
        max_pieces._obj.value = 2 * (z // _cabi.FWD_PIECE) + 1
        build_b._obj.value = 256
        step_d._obj.value = max_pieces._obj.value + 2 * ((n + 255) // 256)
        return 0

    def sdp_forward_build(self, gref, W, g_per_w, p, cell, lam, lam_plane, g, opref, scratch,
                          scratch_bytes, stream):
        d, smin, smax, orders = _grid(gref)
        op = opref._obj
        n = op.n
        strides = np.concatenate([np.cumprod(orders[::-1])[::-1][1:], [1]]).astype(np.int64)
        P = _arr(p, W, ctypes.c_double)
        C = _arr(cell, W * n, ctypes.c_int32).astype(np.int64).reshape(W, n)
        L = np.stack([_arr(lam.value + 8 * k * lam_plane, W * n, ctypes.c_double).reshape(W, n)
                      for k in range(d)])
        x = np.arange(n)
        ys, keys, coefs = [], [], []
        for w in range(W):
            for eps in range(1 << d):
                y = C[w].copy()
                c = np.full(n, P[w])
                for k in range(d):
                    bit = (eps >> k) & 1
                    y += bit * strides[k]
                    c = c * (L[k, w] if bit else 1.0 - L[k, w])
                ys.append(y)
                keys.append(((x * W + w) << d) + eps)
                coefs.append(c)
        y, key, coef = np.concatenate(ys), np.concatenate(keys), np.concatenate(coefs)
        order = np.lexsort((key, y))
        counts = np.bincount(y, minlength=n)
        row_ptr = np.concatenate([[0], np.cumsum(counts)])
        _arr(op.row_ptr, n + 1, ctypes.c_int64)[:] = row_ptr
        _arr(op.src, op.nnz, ctypes.c_int32)[:] = (key[order] >> d) // W
        _arr(op.coef, op.nnz, ctypes.c_double)[:] = coef[order]
        Gv = _arr(g, (W if g_per_w else 1) * n, ctypes.c_double).reshape(-1, n)
        gbar = np.zeros(n)
        for w in range(W):
            gbar = gbar + P[w] * Gv[w if g_per_w else 0]
        _arr(op.gbar, n, ctypes.c_double)[:] = gbar
        npieces = np.where(counts > _cabi.FWD_PIECE, -(-counts // _cabi.FWD_PIECE), 0)
        piece_first = np.concatenate([[0], np.cumsum(npieces)])
        _arr(op.piece_first, n + 1, ctypes.c_int64)[:] = piece_first
        _arr(op.piece_row, op.max_pieces, ctypes.c_int32)[:piece_first[-1]] = np.repeat(x, npieces)
        self.launches += 1
        return 0

    def sdp_forward_steps(self, opref, mu_a, mu_b, n_steps, cost, resid, hist, scratch, stream):
        op = opref._obj
        n, nnz = op.n, op.nnz
        row_ptr = _arr(op.row_ptr, n + 1, ctypes.c_int64)
        dst = np.repeat(np.arange(n), np.diff(row_ptr))
        src = _arr(op.src, nnz, ctypes.c_int32)
        coef = _arr(op.coef, nnz, ctypes.c_double)
        gbar = _arr(op.gbar, n, ctypes.c_double)
        A, B = _arr(mu_a, n, ctypes.c_double), _arr(mu_b, n, ctypes.c_double)
        H = _arr(hist, (n_steps + 1) * n, ctypes.c_double).reshape(-1, n) if (hist.value or 0) else None
        if H is not None:
            H[0] = A
        cin, cout = A, B
        for k in range(n_steps):
            new = np.bincount(dst, weights=coef * cin[src], minlength=n)
            _arr(cost, n_steps, ctypes.c_double)[k] = np.dot(cin, gbar)
            if k + 1 == n_steps and (resid.value or 0):
                _arr(resid, 1, ctypes.c_double)[0] = np.abs(new - cin).sum()
            cout[:] = new
            if H is not None:
                H[k + 1] = new
            cin, cout = cout, cin
        self.launches += 3 * n_steps
        return 0


class _Api(object):
    def __init__(self, pkg, backend):
        self.pkg = pkg
        self.backend = backend
        self.SysDescription = pkg.SysDescription

    def DPSolver(self, sys, **kw):
        if self.backend == "model":
            kw["_test_lib"] = ForwardFakeLib()
        return self.pkg.DPSolver(sys, **kw)


@pytest.fixture(scope="module", params=[pytest.param("model", id="model"),
                                        pytest.param("cuda", marks=gpu, id="cuda")])
def api(request, product):
    return _Api(product, request.param)


@pytest.fixture(scope="module")
def cuda_api(product):
    return _Api(product, "cuda")


# ---------------------------------------------------------------------------
# oracle: P as a scipy.sparse matrix, built from dyn/cost and the oracle's cell search
# ---------------------------------------------------------------------------
def oracle_chain(solver, pol, t_k=None):
    """(P [N x N] csr, g_bar [N]) of the policy `pol` (state_dims + (nc,)) at instant t_k; the
    perturbation nodes are those of the product of all the perturbation grids"""
    sys = solver.sys
    grids = [np.asarray(g, dtype=float) for g in solver.state_grid]
    dims = tuple(len(g) for g in grids)
    n, d = int(np.prod(dims)), len(dims)
    mesh = [m.reshape(n, 1) for m in np.meshgrid(*grids, indexing="ij")]
    u = [pol[..., i].reshape(n, 1) for i in range(pol.shape[-1])]
    if len(solver.perturb_grid):
        # several perturbations: the C-order product of their grids, each passed as a flat (1, W)
        # row, with the products of the marginal probabilities as the joint law
        ws = np.meshgrid(*[np.asarray(g, dtype=float) for g in solver.perturb_grid], indexing="ij")
        ps = np.meshgrid(*[np.asarray(q, dtype=float) for q in solver.perturb_proba], indexing="ij")
        w_args = tuple(w.reshape(1, -1) for w in ws)
        p = np.prod(ps, axis=0).reshape(-1)
    else:
        w_args, p = (), np.ones(1)
    W = len(p)
    args = ((t_k,) if t_k is not None else ()) + tuple(mesh) + tuple(u) + w_args
    nxt = [np.broadcast_to(np.asarray(c, dtype=float), (n, W)) for c in sys.dyn(*args, **sys.params)]
    g = np.broadcast_to(np.asarray(sys.cost(*args, **sys.params), dtype=float), (n, W))
    S = np.stack([c.T.reshape(-1) for c in nxt])           # [d][W*n], w-major
    cell, lam = oc.cell_search([a[0] for a in grids], [a[-1] for a in grids], np.array(dims), S)
    strides = [int(np.prod(dims[k + 1:])) for k in range(d)]
    rows, cols, vals = [], [], []
    xs = np.tile(np.arange(n), W)
    pw = np.repeat(p, n)
    for eps in range(1 << d):
        y = cell.astype(np.int64)
        c = pw.copy()
        for k in range(d):
            bit = (eps >> k) & 1
            y = y + bit * strides[k]
            c = c * (lam[k] if bit else 1 - lam[k])
        rows.append(xs)
        cols.append(y)
        vals.append(c)
    P = sp.csr_matrix((np.concatenate(vals), (np.concatenate(rows), np.concatenate(cols))), shape=(n, n))
    return P, (g * p).sum(axis=1)


def oracle_propagate(solver, pol, mu0, n_steps, time_dependent=False):
    mu = np.asarray(mu0, dtype=float).reshape(-1)
    costs = []
    chain = None if time_dependent else oracle_chain(solver, pol)
    for k in range(n_steps):
        P, gbar = oracle_chain(solver, pol[k], t_k=k) if time_dependent else chain
        costs.append(float(np.dot(mu, gbar)))
        mu = P.T @ mu
    return mu, np.array(costs)


def rel_l1(a, b):
    a, b = np.asarray(a, dtype=float).reshape(-1), np.asarray(b, dtype=float).reshape(-1)
    return float(np.abs(a - b).sum() / max(np.abs(b).sum(), 1e-300))


def _mu0(shape, seed=0):
    return np.random.default_rng(seed).random(shape)


# ---------------------------------------------------------------------------
# the cases
# ---------------------------------------------------------------------------
def _case(api, which):
    """(solver, pol, n_steps, time_dependent)"""
    import workloads as wl
    if which == "inventory":                               # d = 1, W = 4
        prob = wl.inventory(api)
        return prob.solver, golden("inventory.npz")["pol"][5], 20, False
    if which == "ar1_70x5":                                # layout-CF column case, W = 9
        from golden_cases import column_cases
        ar1, _ = column_cases(api)
        return ar1.solver, golden("column_cases.npz")["ar1_pi_pol"], 30, False
    if which == "searev_small":                            # d = 3
        prob = wl.searev(api, n_E=7, n_S=11, n_A=11)
        prob.solver.control_steps = (.01,)
        return prob.solver, golden("searev_small.npz")["pi_pol"], 25, False
    if which == "pv_storage":                              # deterministic, time-dependent, T = 240
        prob = wl.pv_storage(api)
        return prob.solver, golden("pv_storage.npz")["pol"], 240, True
    raise KeyError(which)


CASES = ["inventory", "ar1_70x5", "searev_small", "pv_storage"]


@pytest.mark.parametrize("which", CASES)
def test_propagate_against_scipy_oracle(api, which):
    solver, pol, n_steps, td = _case(api, which)
    mu0 = _mu0(solver._state_grid_shape)
    mu, cost = solver.propagate_distribution(pol, mu0, n_steps=None if td else n_steps, report_time=False)
    mu_o, cost_o = oracle_propagate(solver, pol, mu0, n_steps, td)
    assert mu.shape == solver._state_grid_shape and cost.shape == (n_steps,)
    assert rel_l1(mu, mu_o) <= RTOL
    assert rel_l1(cost, cost_o) <= RTOL
    # history: mu_0 .. mu_n, the last one is the plain result
    m = min(n_steps, 5)
    hist, cost_h = solver.propagate_distribution(pol, mu0, n_steps=m, history=True, report_time=False)
    assert hist.shape == (m + 1,) + solver._state_grid_shape
    assert np.array_equal(hist[0], mu0)
    mu_m, cost_m = solver.propagate_distribution(pol, mu0, n_steps=m, report_time=False)
    assert np.array_equal(hist[-1], mu_m) and np.array_equal(cost_h, cost_m)
    assert rel_l1(hist[m], oracle_propagate(solver, pol, mu0, m, td)[0]) <= RTOL


def test_argument_checks(api):
    solver, pol, _, _ = _case(api, "ar1_70x5")
    dims = solver._state_grid_shape
    mu0 = np.ones(dims)
    with pytest.raises(ValueError, match=r"array `pol` should be of shape"):
        solver.propagate_distribution(pol[..., :1], mu0, n_steps=2, report_time=False)
    with pytest.raises(ValueError, match=r"array `mu0` should be of shape"):
        solver.propagate_distribution(pol, mu0.T, n_steps=2, report_time=False)
    bad = mu0.copy()
    bad[3, 2] = np.nan
    with pytest.raises(ValueError, match="finite"):
        solver.propagate_distribution(pol, bad, n_steps=2, report_time=False)
    bad[3, 2] = np.inf
    with pytest.raises(ValueError, match="finite"):
        solver.stationary_distribution(pol, bad, report_time=False)
    with pytest.raises(ValueError, match="n_steps"):
        solver.propagate_distribution(pol, mu0, report_time=False)
    with pytest.raises(ValueError, match=r"array `pol` should be of shape"):
        solver.stationary_distribution(pol[:, :-1], report_time=False)
    # time-dependent system
    tsolver, tpol, T, _ = _case(api, "pv_storage")
    tmu0 = np.ones(tsolver._state_grid_shape)
    with pytest.raises(ValueError, match="stationary"):
        tsolver.stationary_distribution(tpol[0], report_time=False)
    with pytest.raises(ValueError, match="exceeds"):
        tsolver.propagate_distribution(tpol[:10], tmu0, n_steps=11, report_time=False)
    with pytest.raises(ValueError, match=r"array `pol` should be of shape"):
        tsolver.propagate_distribution(tpol[0], tmu0, report_time=False)


def test_eval_policy_still_refuses_deterministic_systems(api):
    solver, pol, _, _ = _case(api, "pv_storage")
    with pytest.raises(IndexError):
        solver.eval_policy(pol[0], 3, report_time=False)


def test_stationary_distribution_small(api):
    """inventory: a small ergodic chain; pi against scipy's eigenvector of P^T for eigenvalue 1"""
    solver, pol, _, _ = _case(api, "inventory")
    pi, info = solver.stationary_distribution(pol, tol=1e-13, check_every=10, report_time=False)
    P, gbar = oracle_chain(solver, pol)
    mu = np.full(pi.size, 1.0 / pi.size)
    for _ in range(info["n_steps"]):
        mu = P.T @ mu
    assert info["converged"] and len(info["residuals"]) == -(-info["n_steps"] // 10)
    assert info["residuals"][-1] <= 1e-13
    assert rel_l1(pi, mu) <= 1e-12
    assert abs(info["average_cost"] - np.dot(mu, gbar)) <= 1e-12 * abs(np.dot(mu, gbar))
    assert abs(info["mass"] - 1) <= 1e-12 and info["negative_mass"] <= 0
    # an iteration cap returns converged=False without raising
    _, info2 = solver.stationary_distribution(pol, tol=0.0, max_iter=7, check_every=5, report_time=False)
    assert not info2["converged"] and info2["n_steps"] == 7 and len(info2["residuals"]) == 2


# ---------------------------------------------------------------------------
# GPU: full-size operator, duality with eval_policy / bellman_recursion, gain, determinism
# ---------------------------------------------------------------------------
@gpu
def test_config5_three_steps_against_scipy(cuda_api):
    import workloads as wl
    prob = wl.storage_ar1_large(cuda_api)
    _, pol = prob.solver.value_iteration(prob.J0, report_time=False)
    mu0 = _mu0(prob.solver._state_grid_shape, seed=5)
    mu, cost = prob.solver.propagate_distribution(pol, mu0, n_steps=3, report_time=False)
    mu_o, cost_o = oracle_propagate(prob.solver, pol, mu0, 3)
    assert rel_l1(mu, mu_o) <= RTOL and rel_l1(cost, cost_o) <= RTOL


def _ar1_golden(api):
    import workloads as wl
    return wl.storage_ar1(api).solver, golden("storage_ar1.npz")["pi_pol"]


def _searev_golden(api):
    import workloads as wl
    return wl.searev(api).solver, golden("searev_full.npz")["pi_pol"]


@gpu
@pytest.mark.parametrize("which,n", [("storage_ar1", 50), ("searev_full", 200)])
def test_duality_with_eval_policy(cuda_api, which, n):
    solver, pol = (_ar1_golden if which == "storage_ar1" else _searev_golden)(cuda_api)
    mu0 = np.random.default_rng(42).random(solver._state_grid_shape)
    J_n = solver.eval_policy(pol, n, J_zero=np.zeros(solver._state_grid_shape), report_time=False)
    _, cost = solver.propagate_distribution(pol, mu0, n_steps=n, report_time=False)
    fwd, bwd = float(cost.sum()), float(np.dot(mu0.reshape(-1), J_n.reshape(-1)))
    assert abs(fwd - bwd) <= 1e-11 * abs(bwd), (fwd, bwd)


@gpu
def test_time_dependent_duality_with_the_reference_recursion(cuda_api):
    """the reference's own bellman_recursion output (J_fin = 0): <mu_0, J[0]> = sum_k c_k"""
    import workloads as wl
    G = golden("pv_storage.npz")
    solver = wl.pv_storage(cuda_api).solver
    mu0 = np.random.default_rng(7).random(solver._state_grid_shape)
    _, cost = solver.propagate_distribution(G["pol"], mu0, report_time=False)
    fwd, bwd = float(cost.sum()), float(np.dot(mu0, G["J"][0]))
    assert cost.shape == (240,)
    assert abs(fwd - bwd) <= 1e-11 * abs(bwd), (fwd, bwd)


@gpu
def test_gain_of_the_searev_policy(cuda_api):
    """<pi, g_bar> is the gain that relative DP's J_ref converges to; the bound is that
    iteration's own convergence, |J_ref(n) - J_ref(2n)|, plus a rounding floor"""
    G = golden("searev_full.npz")
    solver, pol = _searev_golden(cuda_api)
    pi, info = solver.stationary_distribution(pol, tol=1e-12, max_iter=200_000, report_time=False)
    n = 500
    _, jr_n = solver.eval_policy(pol, n, rel_dp=True, report_time=False)
    _, jr_2n = solver.eval_policy(pol, 2 * n, rel_dp=True, report_time=False)
    bound = abs(jr_n - jr_2n) + 1e-9 * abs(jr_2n)
    print("gain", info["average_cost"], "J_ref(n)", jr_n, "J_ref(2n)", jr_2n, "reference", float(G["pi_Jref"]),
          "steps", info["n_steps"], "converged", info["converged"], "negative mass", info["negative_mass"])
    assert info["converged"]
    assert abs(info["average_cost"] - jr_2n) <= bound
    assert abs(info["average_cost"] - float(G["pi_Jref"])) <= bound
    assert abs(info["mass"] - 1) <= 1e-10


@gpu
def test_mass_conservation_and_determinism(cuda_api):
    solver, pol = _ar1_golden(cuda_api)
    mu0 = np.random.default_rng(3).random(solver._state_grid_shape)
    n = 200
    mu, cost = solver.propagate_distribution(pol, mu0, n_steps=n, report_time=False)
    assert abs(mu.sum() - mu0.sum()) <= 1e-12 * n * mu0.sum()
    mu2, cost2 = solver.propagate_distribution(pol, mu0, n_steps=n, report_time=False)
    assert np.array_equal(mu.view(np.int64), mu2.view(np.int64))
    assert np.array_equal(cost.view(np.int64), cost2.view(np.int64))
    pi, info = solver.stationary_distribution(pol, max_iter=2000, check_every=100, report_time=False)
    pi2, info2 = solver.stationary_distribution(pol, max_iter=2000, check_every=100, report_time=False)
    assert np.array_equal(pi.view(np.int64), pi2.view(np.int64))
    assert info["residuals"] == info2["residuals"] and info["average_cost"] == info2["average_cost"]
