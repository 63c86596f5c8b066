"""Parity of the solver (through the C ABI) against the oracle and the golden
fixtures generated from the unmodified reference.

Solver-level tests run twice: with backend "cuda" (marked gpu: the real
libsdp_b200.so on a B200 - the parity tests proper) and with backend "model"
(CPU suite: the same host code driving tests/fake_lib.py, a numpy model of the
C ABI, so that descriptors, table layout, work items and the argmin -> control
value mapping are checked without a GPU).  Raw-kernel tests are gpu-only.

Bars (BASELINE.json north_star): control policies bit-exact (exact ties are
resolved by the first-minimum rule on both sides; states where the two sides
pick different controls are counted, and must be explainable as near-ties, i.e.
the oracle's J at the two controls differs by <= a few ulp); J within 1e-10
relative in fp64; integer cell indices and fp64 weights bit-exact.
"""
import ctypes
import itertools

import numpy as np
import pytest

from conftest import golden, rel_err, policy_mismatch_report

J_RTOL = 1e-10

gpu = pytest.mark.gpu


class _Api(object):
    """`api` for the workload factories: the product's classes, with the solver
    bound either to the CUDA library or to the numpy model of the C ABI, and
    pinned to one table layout."""

    def __init__(self, pkg, backend, layout="auto", tabulate="auto", compress="auto", column="auto"):
        self.pkg = pkg
        self.backend = backend
        self.layout = layout
        self.tabulate = tabulate
        self.compress = compress
        self.column = column
        self.SysDescription = pkg.SysDescription

    def DPSolver(self, sys, **kw):
        if self.backend == "model":
            from fake_lib import FakeLib
            kw["_test_lib"] = FakeLib()
        sv = self.pkg.DPSolver(sys, **kw)
        sv.table_layout = self.layout
        sv.tabulate = self.tabulate
        sv.table_compress = self.compress
        sv.column_hoist = self.column
        return sv


@pytest.fixture(scope="module", params=[
    pytest.param(("model", "control_minor", "auto", "off"), id="model-A"),
    pytest.param(("model", "state_minor", "auto", "off"), id="model-B"),
    pytest.param(("model", "control_minor", "auto", "auto"), id="model-AF"),
    pytest.param(("model", "state_minor", "auto", "auto", "off"), id="model-BF"),
    pytest.param(("model", "state_minor", "auto", "auto", "auto"), id="model-CF"),
    pytest.param(("cuda", "control_minor", "auto", "off"), marks=gpu, id="cuda-A"),
    pytest.param(("cuda", "state_minor", "auto", "off"), marks=gpu, id="cuda-B"),
    pytest.param(("cuda", "control_minor", "auto", "auto"), marks=gpu, id="cuda-AF"),
    pytest.param(("cuda", "state_minor", "auto", "auto", "off"), marks=gpu, id="cuda-BF"),
    pytest.param(("cuda", "state_minor", "auto", "auto", "auto"), marks=gpu, id="cuda-CF")])
def api(request, product):
    """host logic is exercised against the numpy model of the C ABI (CPU suite)
    and against the real CUDA library (GPU suite), for both table layouts, with
    dense tables (A, B) and with factored tables wherever the system has the
    (x,u) + (x,w) structure (AF, BF; other systems fall back to dense), and with the
    column-shared hoist on top of BF wherever it applies (CF: the storage-AR1 problems,
    whose 41 rows of axis 0 make two tiles per column)"""
    return _Api(product, *request.param)


@pytest.fixture(scope="module")
def cuda_api(product):
    return _Api(product, "cuda")


@pytest.fixture(scope="module")
def eng(product):
    from stodynprog_b200.engine import Engine
    return Engine()


def _adversarial(lo, hi, n, rng):
    span = hi - lo
    x = lo + span * (rng.random(n) * 1.6 - 0.3)
    special = np.array([lo, hi, np.nextafter(hi, lo), np.nextafter(lo, hi), lo - 0.5 * span,
                        hi + 7.3 * span, 3e9, -3e9, 1e300, -1e300, 1e6, np.inf, -np.inf, np.nan,
                        0.0, -0.0, 5e-324, 2147483647.5 * span, -2147483648.5 * span])
    x[:len(special)] = special
    rng.shuffle(x)
    return x


# ---------------------------------------------------------------------------
# K0: cell search, bit-exact
# ---------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("d", [1, 2, 3, 4])
def test_cell_setup_bit_exact(eng, d):
    import torch
    from oracle import oracle as oc
    from stodynprog_b200 import _cabi
    rng = np.random.default_rng(100 + d)
    orders = [(9,), (41, 61), (31, 61, 61), (5, 7, 6, 4)][d - 1]
    smin = np.array([0.0, -4.0, -0.908, 1.5][:d])
    smax = np.array([10.0, 4.0, 0.908, 2.25][:d])
    n = 20000
    s = np.stack([_adversarial(smin[k], smax[k], n, rng) for k in range(d)])
    cell_o, lam_o = oc.cell_search(smin, smax, orders, s)
    grid = _cabi.make_grid([np.linspace(smin[k], smax[k], orders[k]) for k in range(d)])
    s_dev = eng.to_device(s)
    cell = torch.empty(n, dtype=torch.int32, device=eng.device)
    lam = torch.empty(d * n, dtype=torch.float64, device=eng.device)
    rc = eng.lib.sdp_cell_setup(ctypes.byref(grid), n, eng._ptr(s_dev), eng._ptr(cell), eng._ptr(lam),
                                eng.stream)
    _cabi.check(rc, "sdp_cell_setup")
    assert np.array_equal(cell.cpu().numpy(), cell_o)
    lam_g = lam.cpu().numpy().reshape(d, n)
    # bit-exact (NaN payloads excepted)
    assert np.array_equal(np.isnan(lam_g), np.isnan(lam_o))
    ok = ~np.isnan(lam_o)
    assert np.array_equal(lam_g.view(np.int64)[ok], lam_o.view(np.int64)[ok])


# ---------------------------------------------------------------------------
# K2: interpolation
# ---------------------------------------------------------------------------
def _interp_on_path(product, path, monkeypatch, *args):
    """multilinear_interpolation through the host routine (path "host": no launch) or the K2
    kernel (path "device": HOST_MAX_POINTS set to 0), checked by the launch counter, so that a
    change in the routing fails instead of hiding a path"""
    from stodynprog_b200 import _cabi
    if path == "device":
        monkeypatch.setattr(product.interp, "HOST_MAX_POINTS", 0)
    else:
        assert args[3].shape[0] * args[4].shape[1] <= product.interp.HOST_MAX_POINTS
    lib = _cabi.load_library()
    n0 = lib.sdp_launch_count()
    out = product.multilinear_interpolation(*args)
    assert (lib.sdp_launch_count() > n0) == (path == "device")
    return out


@gpu
@pytest.mark.parametrize("d", [1, 2, 3, 4])
@pytest.mark.parametrize("path", ["host", "device"])
def test_interp_golden_bit_exact(product, path, d, monkeypatch):
    """against outputs of the reference's compiled Cython routine"""
    G = golden("interp_kat.npz")
    out = _interp_on_path(product, path, monkeypatch, G["d%d_smin" % d], G["d%d_smax" % d], G["d%d_orders" % d],
                          G["d%d_values" % d], G["d%d_s" % d])
    ref = G["d%d_out" % d]
    assert np.array_equal(np.isnan(out), np.isnan(ref))
    ok = ~np.isnan(ref)
    assert np.array_equal(out.view(np.int64)[ok], ref.view(np.int64)[ok])


@gpu
@pytest.mark.parametrize("d", [1, 2, 3, 4])
@pytest.mark.parametrize("path", ["host", "device"])
def test_interp_f32_golden(product, path, d, monkeypatch):
    G = golden("interp_kat.npz")
    with np.errstate(over="ignore"):
        s32 = np.ascontiguousarray(G["d%d_s" % d].astype(np.float32))
    out = _interp_on_path(product, path, monkeypatch, G["d%d_smin" % d].astype(np.float32),
                          G["d%d_smax" % d].astype(np.float32), G["d%d_orders" % d],
                          G["d%d_values" % d].astype(np.float32), s32)
    assert out.dtype == np.float32
    ref = G["d%d_out_f32" % d]
    # NaN payloads are not part of the contract (x86 makes 0xFFC00000, CUDA's
    # cvt.f32.f64 makes 0x7FFFFFFF): same NaN positions, every other bit equal
    assert np.array_equal(np.isnan(out), np.isnan(ref))
    ok = ~np.isnan(ref)
    assert np.array_equal(out.view(np.int32)[ok], ref.view(np.int32)[ok])


@gpu
def test_interp_1D_reference_kat(product):
    """the reference's own known-answer test (tests/test_dolointerp.py:17-40)"""
    smin, smax, orders = np.array([0.]), np.array([2.]), np.array([3])
    grid = np.linspace(0., 2., 3)
    values = np.ascontiguousarray(np.atleast_2d(grid ** 2))
    pts = np.ascontiguousarray(np.atleast_2d(np.linspace(0., 2., 5)))
    out = product.multilinear_interpolation(smin, smax, orders, values, pts)
    assert np.all(np.abs(out - np.array([0, 0.5, 1, 2.5, 4])) < 1e-10)


@gpu
def test_MultilinearInterpolator_R2R2(product):
    """the reference's test_R2R2 (tests/test_dolointerp.py:45-93), seeded"""
    def f(x):
        return np.vstack([np.sqrt(x[0, :] ** 2 + x[1, :] ** 2),
                          np.power(x[0, :] ** 3 + x[1, :] ** 3, 1.0 / 3.0)])
    interp = product.MultilinearInterpolator([1, 1], [2, 2], [5, 5])
    interp.set_values(f(interp.grid))
    corners = np.array([[1, 1], [1, 2], [2, 1], [2, 2]], dtype=float).T
    rnd = np.random.default_rng(0).random((2, 6)) + 1
    for pts, tol in ((corners, 1e-9), (rnd, 0.01)):
        assert np.all(np.abs(interp(pts) - f(pts)) < tol)


@gpu
def test_interp_on_state_broadcast(product, port):
    import workloads as wl
    prob = wl.storage_ar1(product, n_E=11, n_P=13)
    ora = wl.storage_ar1(port, n_E=11, n_P=13)
    A = np.random.default_rng(3).standard_normal((11, 13))
    f, fo = prob.solver.interp_on_state(A), ora.solver.interp_on_state(A)
    x = np.linspace(-1, 11, 7).reshape(-1, 1)
    y = np.linspace(-5, 5, 5)
    assert f(x, y).shape == (7, 5)
    assert np.array_equal(f(x, y), fo(x, y))
    assert f(0, 0).shape == ()
    with pytest.raises(ValueError):
        prob.solver.interp_on_state(np.zeros((3, 3)))


# ---------------------------------------------------------------------------
# config #1: inventory (doc/example_inventory.rst:217-239 + reference run)
# ---------------------------------------------------------------------------
def test_inventory_golden(api):
    import workloads as wl
    G = golden("inventory.npz")
    prob = wl.inventory(api)
    J = prob.J0
    for k in range(6):
        J, u = prob.solver.value_iteration(J, report_time=False)
        assert u.shape == (10, 1)
        assert np.array_equal(u, G["pol"][k]), "policy after sweep %d" % (k + 1)
        assert rel_err(J, G["J"][k]) <= J_RTOL
        if k == 0:   # printed in the reference's doc
            assert np.allclose(J, [9, 6, 3, 0, .5, 1, 1.5, 2, 2.5, 3], rtol=0, atol=1e-12)
    assert np.array_equal(G["pol"][3][:, 0], [5, 4, 3, 2, 1, 0, 0, 0, 0, 0])


# ---------------------------------------------------------------------------
# config #2: deterministic time-dependent storage, bellman_recursion
# ---------------------------------------------------------------------------
def test_pv_storage_bellman_recursion_vs_port(api, port):
    """short horizon, coarse control step (the model backend is slow)"""
    import workloads as wl
    prob = wl.pv_storage(api, horizon=30)
    prob.solver.control_steps = (.01,)
    J, pol = prob.solver.bellman_recursion(30, prob.J_fin, report_time=False)
    ora = wl.pv_storage(port, horizon=30)
    ora.solver.control_steps = (.01,)
    Jo, polo = ora.solver.bellman_recursion(30, ora.J_fin)
    assert J.shape == (30, 50) and pol.shape == (30, 50, 1)
    n_bad, _ = policy_mismatch_report(pol, polo)
    assert n_bad == 0
    assert rel_err(J, Jo) <= J_RTOL


def test_recursion_fast_path_and_its_refusals(api, port):
    """bellman_recursion: when only the stage cost depends on the instant the tables are built
    once and the sweeps run back to back (Engine.recursion_fast) - same J and policies, bit for
    bit, as the instant-by-instant path; dynamics or admissible controls that do depend on
    the instant are detected and take the instant-by-instant path (and match the port)"""
    import workloads as wl
    out = {}
    for mode in ("auto", "per_instant"):
        prob = wl.pv_storage(api, horizon=12)
        sv = prob.solver
        sv.control_steps = (.02,)
        sv.recursion_mode = mode
        out[mode] = sv.bellman_recursion(12, prob.J_fin, report_time=False)
        assert (sv.last_recursion is not None) == (mode == "auto")
        if mode == "auto":
            assert sv.last_recursion["instants"] == 12
    assert _same_bits(out["auto"][0], out["per_instant"][0]) and np.array_equal(out["auto"][1], out["per_instant"][1])

    def variant(a, what):
        prob = wl.pv_storage(a, horizon=12)
        sv, sysd = prob.solver, prob.sys
        sv.control_steps = (.02,)
        dyn0, box0 = sysd.dyn, sysd.control_box
        if what == "dyn":          # a self-discharge that sets in half-way
            sysd._dyn = lambda k, E, P: (dyn0(k, E, P)[0] - 0.01 * E * (k >= 6),)
        else:                       # the rated power shrinks with the instant
            def box(k, E):
                (lo, hi), = box0(k, E)
                return ((lo * (1 - 0.02 * k), hi),)
            sysd._control_box = box
        return prob
    for what in ("dyn", "box"):
        prob, ora = variant(api, what), variant(port, what)
        J, pol = prob.solver.bellman_recursion(12, prob.J_fin, report_time=False)
        assert prob.solver.last_recursion is None
        Jo, polo = ora.solver.bellman_recursion(12, ora.J_fin)
        assert policy_mismatch_report(pol, polo)[0] == 0 and rel_err(J, Jo) <= J_RTOL


@gpu
def test_pv_storage_full_horizon_golden(cuda_api):
    import workloads as wl
    G = golden("pv_storage.npz")
    prob = wl.pv_storage(cuda_api)
    J, pol = prob.solver.bellman_recursion(prob.horizon, prob.J_fin, report_time=False)
    n_bad, _ = policy_mismatch_report(pol, G["pol"])
    assert n_bad == 0
    assert rel_err(J, G["J"]) <= J_RTOL


# ---------------------------------------------------------------------------
# config #3: storage + AR(1) - the roofline target grid
# ---------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ar1(cuda_api):
    import workloads as wl
    return wl.storage_ar1(cuda_api)


@gpu
def test_storage_ar1_control_counts(ar1):
    """notebook print_summary: [4,001 to 8,001] values, 6,342.5 on average"""
    G = golden("storage_ar1.npz")
    T = ar1.solver.sweep_tables()
    assert np.array_equal(T.host_full.npts, G["control_dims"])
    assert T.host_full.npts[:, 0].min() == 4001 and T.host_full.npts[:, 0].max() == 8001
    assert abs(T.host_full.npts[:, 0].mean() - 6342.5) < 0.05
    assert T.n_backups_total == 142762509


@gpu
def test_storage_ar1_value_iteration_golden(ar1):
    G = golden("storage_ar1.npz")
    J = ar1.J0
    for k in range(3):
        J, pol = ar1.solver.value_iteration(J, report_time=False)
        n_bad, _ = policy_mismatch_report(pol, G["vi_pol%d" % k])
        assert n_bad == 0, "sweep %d: %d states with a different control" % (k, n_bad)
        assert rel_err(J, G["vi_J%d" % k]) <= J_RTOL


@gpu
def test_storage_ar1_eval_policy_golden(ar1):
    G = golden("storage_ar1.npz")
    J, J_ref = ar1.solver.eval_policy(G["pol_ini"], 50, rel_dp=True, J_ref_full=True, report_time=False)
    assert rel_err(J_ref, G["ev_Jref_hist"]) <= J_RTOL
    assert np.max(np.abs(J - G["ev_J"])) <= J_RTOL * np.max(np.abs(G["ev_J"]))


@gpu
def test_storage_ar1_policy_iteration_golden(ar1, capsys):
    """notebook golden: 0.105724, 0.0486519, 0.0468464, 0.0468268, 0.0468268"""
    G = golden("storage_ar1.npz")
    (J, J_ref), pol = ar1.solver.policy_iteration(ar1.initial_policy(), 50, 4, rel_dp=True)
    text = capsys.readouterr().out
    costs = [l.split(':')[1].strip() for l in text.splitlines() if 'ref policy cost' in l]
    assert costs == ['0.105724', '0.0486519', '0.0468464', '0.0468268', '0.0468268']
    assert abs(J_ref - float(G["pi_Jref"])) <= J_RTOL * abs(float(G["pi_Jref"]))
    n_bad, _ = policy_mismatch_report(pol, G["pi_pol"])
    assert n_bad == 0
    assert np.max(np.abs(J - G["pi_J"])) <= J_RTOL * np.max(np.abs(G["pi_J"]))


@gpu
def test_storage_ar1_random_J_vs_port(ar1, port):
    """non-trivial J (no ties): argmin index and J against the numpy port on a
    subset of states, plus exact agreement with the ordered-sum C oracle."""
    import workloads as wl
    ora = wl.storage_ar1(port)
    J0 = np.random.default_rng(0).standard_normal((41, 61))
    J, pol = ar1.solver.value_iteration(J0, report_time=False)
    lo, hi = 1000, 1120
    Jo, polo = ora.solver.value_iteration(J0, state_slice=(lo, hi))
    sl = slice(lo, hi)
    assert np.array_equal(pol.reshape(-1, 2)[sl], polo.reshape(-1, 2)[sl])
    assert rel_err(J.reshape(-1)[sl], Jo.reshape(-1)[sl]) <= J_RTOL


@gpu
def test_storage_ar1_sup_norm_and_device_loop(ar1):
    J, pol, info = ar1.solver.solve_value_iteration(max_iter=3, tol=0.0)
    G = golden("storage_ar1.npz")
    assert info["n_sweeps"] == 3
    assert rel_err(J, G["vi_J2"]) <= J_RTOL
    n_bad, _ = policy_mismatch_report(pol, G["vi_pol2"])
    assert n_bad == 0
    r_expected = np.max(np.abs(G["vi_J2"] - G["vi_J1"]))
    assert abs(info["residuals"][-1] - r_expected) <= 1e-9 * r_expected


def test_item_chunking_invariance(api):
    """splitting a state's controls into runs must not change anything"""
    import workloads as wl
    J0 = np.random.default_rng(5).standard_normal((9, 11))
    res = []
    for chunk in (64, 512, 100000):
        prob = wl.storage_ar1(api, n_E=9, n_P=11, steps=(0.01, 0.1), item_chunk=chunk)
        res.append(prob.solver.value_iteration(J0, report_time=False))
    for J, pol in res[1:]:
        assert np.array_equal(J, res[0][0]) and np.array_equal(pol, res[0][1])


# ---------------------------------------------------------------------------
# config #4: SEAREV (3-D)
# ---------------------------------------------------------------------------
def _searev_small(api, **kw):
    import workloads as wl
    prob = wl.searev(api, n_E=7, n_S=11, n_A=11, **kw)
    prob.solver.control_steps = (.01,)
    return prob


def test_searev_small_golden(api):
    G = golden("searev_small.npz")
    prob = _searev_small(api)
    J = prob.J0
    for k in range(2):
        J, pol = prob.solver.value_iteration(J, report_time=False)
        n_bad, _ = policy_mismatch_report(pol, G["vi_pol%d" % k])
        assert n_bad == 0
        assert rel_err(J, G["vi_J%d" % k]) <= J_RTOL
    (Jd, Jr), pol = prob.solver.policy_iteration(prob.initial_policy(), 30, 2, rel_dp=True)
    n_bad, _ = policy_mismatch_report(pol, G["pi_pol"])
    assert n_bad == 0
    assert abs(Jr - float(G["pi_Jref"])) <= J_RTOL * abs(float(G["pi_Jref"]))
    assert np.max(np.abs(Jd - G["pi_J"])) <= J_RTOL * np.max(np.abs(G["pi_J"]))


# ---------------------------------------------------------------------------
# semantics: ties, NaN, deterministic branch, w-dependent cost, 4-D state
# ---------------------------------------------------------------------------
def _toy(api, d=1, cost_kind="plain", n_u=37, n_w=5, **kw):
    """small synthetic system exercising the generic paths; n_w perturbation nodes on
    [-0.9, 0.9], or none (a deterministic system) with n_w = 0"""
    import scipy.stats as stats

    def dyn(*a):
        x, (u, w) = a[:d], a[d:]
        return tuple(0.9 * xi + (0.3 + 0.1 * i) * u + (0.5 if i == d - 1 else 0.0) * w
                     for i, xi in enumerate(x))

    def box(*x):
        return ((-1.0 - 0.1 * x[0], 1.0 + 0.05 * x[0]),)

    def cost(*a):
        x, (u, w) = a[:d], a[d:]
        base = sum(xi ** 2 for xi in x) + 0.1 * u ** 2
        if cost_kind == "w":
            return base + 0.05 * w * u
        if cost_kind == "flat":
            return 0. * u + 1.0        # every control ties exactly
        if cost_kind == "nan":
            return np.where((u > 0.2) & (u < 0.4), np.nan, base)
        return base

    names = ['x%d' % i for i in range(d)]
    w_arg, w_val = (", w", "w") if n_w else ("", "0.0")
    src = "def dyn_f({0}, u{1}): return dyn({0}, u, {2})\n" \
          "def cost_f({0}, u{1}): return cost({0}, u, {2})\n" \
          "def box_f({0}): return box({0})\n".format(', '.join(names), w_arg, w_val)
    ns = {'dyn': dyn, 'cost': cost, 'box': box}
    exec(src, ns)
    sys = api.SysDescription((d, 1, 1 if n_w else 0), name='toy%d' % d)
    sys.dyn = ns['dyn_f']
    sys.control_box = ns['box_f']
    sys.cost = ns['cost_f']
    if n_w:
        sys.perturb_laws = [stats.norm(0, 0.3)]
    sv = api.DPSolver(sys, **kw)
    sizes = [6, 5, 4, 3][:d]
    args = []
    for n in sizes:
        args += [-1.0, 2.0, n]
    sv.discretize_state(*args)
    if n_w:
        sv.discretize_perturb(-0.9, 0.9, n_w)
    sv.control_steps = (2.0 / n_u,)
    return sv


@pytest.mark.parametrize("d", [1, 2, 3, 4])
@pytest.mark.parametrize("cost_kind", ["plain", "w", "flat", "nan"])
def test_toy_systems_vs_port(api, port, d, cost_kind):
    sv, so = _toy(api, d, cost_kind), _toy(port, d, cost_kind)
    shape = sv._state_grid_shape
    J0 = np.random.default_rng(d).standard_normal(shape)
    J, pol = sv.value_iteration(J0, report_time=False)
    with np.errstate(invalid="ignore"):
        Jo, polo, idxo = so.value_iteration(J0, want_index=True)
    assert np.array_equal(pol, polo)
    both_nan = np.isnan(J) & np.isnan(Jo)
    assert np.array_equal(np.isnan(J), np.isnan(Jo))
    assert rel_err(np.where(both_nan, 0, J), np.where(both_nan, 0, Jo)) <= J_RTOL
    assert sv.last_tables.g_per_w == (1 if cost_kind == "w" else 0)
    assert sv.last_tables.tiled == (sv.table_layout == "state_minor")
    # policy evaluation of the greedy policy, with and without relative DP
    if cost_kind != "nan":
        Je = sv.eval_policy(pol, 7, report_time=False)
        Jeo = so.eval_policy(polo, 7)
        assert rel_err(Je, Jeo) <= J_RTOL
        Jr, ref = sv.eval_policy(pol, 7, rel_dp=True, report_time=False)
        Jro, refo = so.eval_policy(polo, 7, rel_dp=True)
        assert abs(ref - refo) <= J_RTOL * abs(refo)
        assert np.max(np.abs(Jr - Jro)) <= J_RTOL * max(np.max(np.abs(Jro)), 1e-300)


def _two_perturbations(api, kind, n0=6, **kw):
    """2 states, 1 control, TWO perturbations (a continuous one on 3 nodes, a discrete one on 2):
    `kind` "mixed": a coordinate and the cost depend on control AND perturbations (dense tables);
    "split": E-like coordinate follows the control, the other the perturbations (factored)"""
    import scipy.stats as stats

    def dyn(x0, x1, u, w1, w2):
        if kind == "mixed":
            return (0.9 * x0 + 0.4 * u + 0.3 * w1, 0.8 * x1 + 0.2 * u * w2 + 0.1 * w1)
        return (x0 + 0.5 * u, 0.8 * x1 + 0.3 * w1 + 0.25 * w2)

    def box(x0, x1):
        return ((-1.0 - 0.1 * x0, 1.0 + 0.05 * x0),)

    def cost(x0, x1, u, w1, w2):
        base = x0 ** 2 + 0.5 * x1 ** 2 + 0.1 * u ** 2
        return base + 0.05 * w1 * u - 0.02 * w2 if kind == "mixed" else base

    sys = api.SysDescription((2, 1, 2), name='two perturbations')
    sys.dyn, sys.control_box, sys.cost = dyn, box, cost
    sys.perturb_laws = [stats.norm(0, 0.5), stats.rv_discrete(values=([0, 1], [0.3, 0.7])).freeze()]
    sv = api.DPSolver(sys, **kw)
    sv.discretize_state(-1.0, 2.0, n0, -1.0, 1.5, 5)
    sv.discretize_perturb(-0.9, 0.9, 3, 0, 1, 2)
    sv.control_steps = (2.0 / 23,)
    return sv


def test_two_perturbations_port_against_brute_force(port):
    """the oracle port's convention for several perturbations (the reference has a TODO there,
    stodynprog.py:614,666,679-683) pinned against explicit loops: for every control, the sum
    over (w1, w2) in C order of p1[i]*p2[j] * (g + J(f(x, u, w1_i, w2_j)))"""
    from oracle import oracle as oc
    for kind in ("mixed", "split"):
        so = _two_perturbations(port, kind)
        sysd = so.sys
        J0 = np.random.default_rng(5).standard_normal(so._state_grid_shape)
        Jo, polo = so.value_iteration(J0)
        smin = np.array([g[0] for g in so.state_grid])
        smax = np.array([g[-1] for g in so.state_grid])
        orders = np.array([len(g) for g in so.state_grid], dtype=np.int64)
        vals = np.ascontiguousarray(J0.reshape(1, -1))
        (w1, w2), (p1, p2) = so.perturb_grid, so.perturb_proba
        for i0, x0 in enumerate(so.state_grid[0]):
            for i1, x1 in enumerate(so.state_grid[1]):
                (ug,), _ = so.control_grids((x0, x1))
                best, best_u = None, None
                for u in ug:
                    acc = 0.0
                    for a, wa in enumerate(w1):
                        for b, wb in enumerate(w2):
                            xn = sysd.dyn(x0, x1, u, wa, wb)
                            pt = np.array([[float(xn[0])], [float(xn[1])]])
                            v = float(oc.interp(smin, smax, orders, vals, pt)[0, 0])
                            acc += (sysd.cost(x0, x1, u, wa, wb) + v) * (p1[a] * p2[b])
                    if best is None or acc < best:
                        best, best_u = acc, u
                assert abs(Jo[i0, i1] - best) <= 1e-12 * max(abs(best), 1.0)
                assert polo[i0, i1, 0] == best_u


@pytest.mark.parametrize("kind", ["mixed", "split"])
def test_two_perturbations_vs_port(api, port, kind):
    """value iteration, policy evaluation and policy iteration with a product perturbation grid
    (3 x 2 nodes flattened to W = 6) against the oracle port"""
    sv, so = _two_perturbations(api, kind), _two_perturbations(port, kind)
    J0 = np.random.default_rng(6).standard_normal(sv._state_grid_shape)
    J, pol = sv.value_iteration(J0, report_time=False)
    Jo, polo = so.value_iteration(J0)
    T = sv.last_tables
    assert T.W == 6 and T.expect == 1
    assert bool(T.u_mask) == (kind == "split" and sv.table_compress != "off")
    assert np.array_equal(pol, polo) and rel_err(J, Jo) <= J_RTOL
    Je, ref = sv.eval_policy(pol, 6, rel_dp=True, report_time=False)
    Jeo, refo = so.eval_policy(polo, 6, rel_dp=True)
    assert abs(ref - refo) <= J_RTOL * abs(refo) and np.max(np.abs(Je - Jeo)) <= J_RTOL * np.max(np.abs(Jeo))
    (Jp, Jr), polp = sv.policy_iteration(pol, 4, 2, rel_dp=True)
    (Jpo, Jro), polpo = so.policy_iteration(polo, 4, 2, rel_dp=True)
    assert np.array_equal(polp, polpo) and abs(Jr - Jro) <= J_RTOL * abs(Jro)


@pytest.mark.parametrize("backend", [pytest.param("model"), pytest.param("cuda", marks=gpu)])
def test_two_perturbations_column_layout(product, port, backend):
    """the product perturbation grid through layout CF (40 rows of axis 0, W = 6 <= 9 slots)"""
    api = _Api(product, backend, "state_minor", "auto", "on", "on")
    sv, so = _two_perturbations(api, "split", n0=40), _two_perturbations(port, "split", n0=40)
    J0 = np.random.default_rng(7).standard_normal(sv._state_grid_shape)
    J, pol = sv.value_iteration(J0, report_time=False)
    Jo, polo = so.value_iteration(J0)
    assert sv.last_tables.layout_name == "column_factored"
    assert np.array_equal(pol, polo) and rel_err(J, Jo) <= J_RTOL


def test_rel_dp_value_iteration(api, port):
    sv, so = _toy(api, 2), _toy(port, 2)
    J0 = np.zeros(sv._state_grid_shape)
    (Jd, Jr), pol = sv.value_iteration((J0, 0.), rel_dp=True, report_time=False)
    (Jdo, Jro), polo = so.value_iteration((J0, 0.), rel_dp=True)
    assert np.array_equal(pol, polo)
    assert Jd[sv._state_ref_ind] == 0.
    assert abs(Jr - Jro) <= J_RTOL * abs(Jro)
    assert np.max(np.abs(Jd - Jdo)) <= J_RTOL * np.max(np.abs(Jdo))
    with pytest.raises(AssertionError):
        sv.value_iteration((J0 + 1., 0.), rel_dp=True, report_time=False)
    with pytest.raises(ValueError):
        sv.value_iteration(np.zeros((2, 2)), report_time=False)


@gpu
def test_supnorm_kernel(eng):
    import torch
    from stodynprog_b200 import _cabi
    rng = np.random.default_rng(9)
    a = rng.standard_normal(100003)
    b = rng.standard_normal(100003)
    a[17] = np.nan
    out = torch.zeros(1, dtype=torch.float64, device=eng.device)
    ad, bd = eng.to_device(a), eng.to_device(b)
    rc = eng.lib.sdp_supnorm_diff(eng._ptr(ad), eng._ptr(bd), a.size, eng._ptr(out), eng.stream)
    _cabi.check(rc, "sdp_supnorm_diff")
    assert out.cpu().numpy()[0] == np.nanmax(np.abs(a - b))


@gpu
def test_abi_rejects_bad_arguments(eng):
    from stodynprog_b200 import _cabi
    g = _cabi.SdpGrid()
    g.d = 7
    rc = eng.lib.sdp_cell_setup(ctypes.byref(g), 1, None, None, None, None)
    assert rc == -1 and b"grid.d" in eng.lib.sdp_last_error()
    with pytest.raises(_cabi.SdpLibraryError):
        _cabi.check(rc, "sdp_cell_setup")


@gpu
def test_memcpy_2d_and_finalize_cols_through_the_abi(eng, cuda_api):
    """sdp_memcpy_2d: a column range of a C-order device array into the same columns of a
    page-locked host array, nothing else touched; argument checks of the two entry points of the
    column-piece path"""
    import torch
    import workloads as wl
    from stodynprog_b200 import _cabi
    lib = eng.lib
    rows, cols = 37, 23
    src = torch.arange(rows * cols, dtype=torch.float64, device=eng.device)
    dst = torch.full((rows * cols,), -1.0, dtype=torch.float64).pin_memory()
    c0, c1 = 5, 14
    rc = lib.sdp_memcpy_2d(ctypes.c_void_p(dst.data_ptr() + 8 * c0), 8 * cols,
                           ctypes.c_void_p(src.data_ptr() + 8 * c0), 8 * cols, 8 * (c1 - c0), rows, eng.stream)
    _cabi.check(rc, "sdp_memcpy_2d")
    eng.sync()
    want = np.full((rows, cols), -1.0)
    want[:, c0:c1] = np.arange(rows * cols, dtype=float).reshape(rows, cols)[:, c0:c1]
    assert np.array_equal(dst.numpy().reshape(rows, cols), want)
    assert lib.sdp_memcpy_2d(eng._ptr(dst), 8, eng._ptr(src), 8 * cols, 16, rows, eng.stream) == -1
    assert b"sdp_memcpy_2d" in lib.sdp_last_error()
    assert lib.sdp_memcpy_2d(None, 8 * cols, eng._ptr(src), 8 * cols, 8, rows, eng.stream) == -1
    assert lib.sdp_memcpy_2d(eng._ptr(dst), 8 * cols, eng._ptr(src), 8 * cols, 0, rows, eng.stream) == 0
    # finalize_cols: tables that are not in layout CF, a column range outside the grid, missing policy arrays
    sv = wl.storage_ar1(cuda_api, n_E=70, n_P=6, n_w=9, steps=(0.3, 0.1)).solver
    sv.table_layout, sv.column_hoist = "state_minor", "off"
    T = sv.sweep_tables()
    args = (eng._ptr(T.part_val), eng._ptr(T.part_idx), eng._ptr(T.J_out), eng._ptr(T.argmin))
    assert lib.sdp_sweep_finalize_cols(ctypes.byref(T.c_tables), *args, 6, 0, 0, None, None, None, None, 0,
                                       eng.stream) == -1
    assert b"layout CF" in lib.sdp_last_error()
    sv = wl.storage_ar1(cuda_api, n_E=70, n_P=6, n_w=9, steps=(0.3, 0.1)).solver
    sv.table_layout, sv.column_hoist = "state_minor", "on"
    T = sv.sweep_tables()
    assert T.column
    args = (eng._ptr(T.part_val), eng._ptr(T.part_idx), eng._ptr(T.J_out), eng._ptr(T.argmin))
    assert lib.sdp_sweep_finalize_cols(ctypes.byref(T.c_tables), *args, 5, 0, 0, None, None, None, None, 0,
                                       eng.stream) == -1          # 6 columns do not fit a grid of 5
    assert lib.sdp_sweep_finalize_cols(ctypes.byref(T.c_tables), *args, 6, 0, 2, None, None, None, None, 0,
                                       eng.stream) == -1          # nc > 0 without lo / hi / npts / pol
    assert b"sdp_sweep_finalize_cols" in lib.sdp_last_error()


# ---------------------------------------------------------------------------
# host tabulation: one call per chunk of states == one call per state
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("backend", [pytest.param("model"), pytest.param("cuda", marks=gpu)])
@pytest.mark.parametrize("layout", ["control_minor", "state_minor"])
@pytest.mark.parametrize("which", ["storage_ar1", "searev", "toy_w", "curtail"])
def test_batched_tabulation_is_bit_identical(product, backend, layout, which):
    import workloads as wl
    tabs = []
    for mode in ("per_state", "batched"):
        api = _Api(product, backend, layout, mode, "off")
        if which == "storage_ar1":
            sv = wl.storage_ar1(api, n_E=9, n_P=11, steps=(0.01, 0.1)).solver
        elif which == "searev":
            sv = _searev_small(api).solver
        elif which == "toy_w":
            sv = _toy(api, 3, "w")
        else:
            sv = _two_control_system(api)
        T = sv.sweep_tables()
        assert T.tabulate_mode == mode
        tabs.append(T)
    a, b = tabs
    assert a.n_entries == b.n_entries and a.g_per_w == b.g_per_w
    n = a.n_entries
    assert np.array_equal(a.cell[:n].cpu().numpy(), b.cell[:n].cpu().numpy())
    la = a.lam.cpu().numpy().view(np.int64).reshape(a.d, -1)[:, :n]
    lb = b.lam.cpu().numpy().view(np.int64).reshape(b.d, -1)[:, :n]
    assert np.array_equal(la, lb)
    assert np.array_equal(a.g.cpu().numpy().view(np.int64), b.g.cpu().numpy().view(np.int64))


# ---------------------------------------------------------------------------
# factored (x,u) + (x,w) tables: same entries, same sweep, bit for bit
# ---------------------------------------------------------------------------
def _separable(api, roles, n_u=23, n_w=5, **kw):
    """synthetic system whose next-state coordinate k depends on the state and on
    the control only (role 'u'), the perturbation only ('w') or neither ('x')"""
    import scipy.stats as stats
    d = len(roles)

    def dyn(*a):
        x, (u, w) = a[:d], a[d:]
        out = []
        for k, role in enumerate(roles):
            if role == 'u':
                out.append(0.8 * x[k] + (0.4 + 0.1 * k) * u)
            elif role == 'w':
                out.append(0.7 * x[k] + 0.3 * x[0] + (1.0 + 0.2 * k) * w)
            else:
                out.append(0.9 * x[k] + 0.1)
        return tuple(out)

    def box(*x):
        return ((-1.0 - 0.1 * x[0], 1.0 + 0.05 * x[-1]),)

    def cost(*a):
        x, (u, w) = a[:d], a[d:]
        return sum(xi ** 2 for xi in x) + 0.1 * (u - 0.2) ** 2

    names = ['x%d' % i for i in range(d)]
    src = "def dyn_f({0}, u, w): return dyn({0}, u, w)\n" \
          "def cost_f({0}, u, w): return cost({0}, u, w)\n" \
          "def box_f({0}): return box({0})\n".format(', '.join(names))
    ns = {'dyn': dyn, 'cost': cost, 'box': box}
    exec(src, ns)
    sys = api.SysDescription((d, 1, 1), name='separable' + ''.join(roles))
    sys.dyn = ns['dyn_f']
    sys.control_box = ns['box_f']
    sys.cost = ns['cost_f']
    sys.perturb_laws = [stats.norm(0, 0.3)]
    sv = api.DPSolver(sys, **kw)
    args = []
    for n in [7, 6, 5][:d]:
        args += [-1.0, 2.0, n]
    sv.discretize_state(*args)
    sv.discretize_perturb(-0.9, 0.9, n_w)
    sv.control_steps = (2.0 / n_u,)
    return sv


def _dense_from_factored(T):
    """expand factored tables on the host into the dense (cell, lam[d], g) entries,
    in the dense layout's order"""
    W, d, n = T.W, T.d, T.n_states
    ku = [k for k in range(d) if (T.u_mask >> k) & 1]
    kw = [k for k in range(d) if not (T.u_mask >> k) & 1]
    cu = T.cell.cpu().numpy().astype(np.int64)
    lu = T.lam.cpu().numpy().reshape(len(ku), -1)
    g = T.g.cpu().numpy()
    cw = T.cell_w.cpu().numpy().astype(np.int64)
    lw = T.lam_w.cpu().numpy().reshape(len(kw), -1)
    U = T.U_dev.cpu().numpy()[:n]
    cells, lams, gs = [], [[] for _ in range(d)], []
    if not T.tiled:
        Upad = (U + 3) // 4 * 4
        eo = np.concatenate([[0], np.cumsum(Upad)])
        for i in range(n):
            e = slice(eo[i], eo[i] + Upad[i])
            for w in range(W):
                live = np.arange(Upad[i]) < U[i]
                cells.append(np.where(live, cu[e] + cw[i * W + w], 0))
                for j, k in enumerate(ku):
                    lams[k].append(lu[j][e])
                for j, k in enumerate(kw):
                    lams[k].append(np.where(live, lw[j][i * W + w], 0.0))
            gs.append(g[e])
    else:
        n_tiles = (n + 31) // 32
        Ut = np.zeros(n_tiles * 32, dtype=np.int64)
        Ut[:n] = U
        Ulane = Ut.reshape(n_tiles, 32)
        tU = Ulane.max(axis=1)
        to = np.concatenate([[0], np.cumsum(tU * 32)])
        for t in range(n_tiles):
            blk = slice(to[t], to[t] + tU[t] * 32)
            cu_t = cu[blk].reshape(tU[t], 1, 32)
            live = np.arange(tU[t])[:, None, None] < Ulane[t][None, None, :]
            cw_t = cw[t * W * 32:(t + 1) * W * 32].reshape(1, W, 32)
            cells.append(np.where(live, cu_t + cw_t, 0).reshape(-1))
            for j, k in enumerate(ku):
                lams[k].append(np.broadcast_to(lu[j][blk].reshape(tU[t], 1, 32), (tU[t], W, 32)).reshape(-1))
            for j, k in enumerate(kw):
                lw_t = lw[j][t * W * 32:(t + 1) * W * 32].reshape(1, W, 32)
                lams[k].append(np.where(live, lw_t, 0.0).reshape(-1))
            gs.append(g[blk])
    return (np.concatenate(cells), [np.concatenate(l) for l in lams], np.concatenate(gs))


FACTOR_CASES = {
    "storage_ar1": 0b01, "searev": None, "curtail": 0b01, "coarse_controls": 0b01,
    "uw": 0b01, "wu": 0b10, "uww": 0b001, "wuw": 0b010, "uuw": 0b011, "wwu": 0b100,
    "uwu": 0b101, "wuu": 0b110, "xuw": 0b010, "xwu": 0b100,
}


def _factor_case(api, which):
    import workloads as wl
    if which == "storage_ar1":
        return wl.storage_ar1(api, n_E=9, n_P=11, steps=(0.01, 0.1)).solver
    if which == "searev":
        return _searev_small(api).solver
    if which == "curtail":
        return _two_control_system(api)
    if which == "coarse_controls":
        # controls several state-grid rows apart: the per-item inner-interpolation
        # table of the AF kernel does not fit and its generic path runs
        return wl.storage_ar1(api, n_E=150, n_P=7, n_w=5, steps=(8. / 255, 0.1)).solver
    return _separable(api, which)


@pytest.mark.parametrize("backend", [pytest.param("model"), pytest.param("cuda", marks=gpu)])
@pytest.mark.parametrize("layout", ["control_minor", "state_minor"])
@pytest.mark.parametrize("which", sorted(FACTOR_CASES))
def test_factored_tables_and_sweep_equal_dense(product, backend, layout, which):
    """the factored layouts hold exactly the entries of the dense tables (K0) and
    the factored sweep returns bit-identical J and argmin (K1)"""
    dense = _factor_case(_Api(product, backend, layout, "auto", "off"), which)
    fact = _factor_case(_Api(product, backend, layout, "auto", "on"), which)
    fact.column_hoist = "off"         # (layout CF reorders the tiles; it has its own tests)
    Td, Tf = dense.sweep_tables(), fact.sweep_tables()
    assert not Td.factored and Tf.factored
    if FACTOR_CASES[which] is not None:
        assert Tf.u_mask == FACTOR_CASES[which]
    assert Tf.layout_name == layout + "_factored"
    cells, lams, g = _dense_from_factored(Tf)
    n = Td.n_entries
    assert np.array_equal(Td.cell.cpu().numpy()[:n], cells)
    ld = Td.lam.cpu().numpy().reshape(Td.d, -1)[:, :n]
    for k in range(Td.d):
        assert np.array_equal(ld[k].view(np.int64), lams[k].view(np.int64)), k
    assert np.array_equal(Td.g.cpu().numpy()[:len(g)].view(np.int64), g.view(np.int64))
    assert Tf.device_bytes < Td.device_bytes
    J0 = np.random.default_rng(5).standard_normal(dense._state_grid_shape)
    for _ in range(2):
        Jd, pold = dense.value_iteration(J0, report_time=False)
        Jf, polf = fact.value_iteration(J0, report_time=False)
        assert np.array_equal(Jd.view(np.int64), Jf.view(np.int64))
        assert np.array_equal(pold, polf)
        J0 = Jd


@gpu
@pytest.mark.parametrize("which", ["storage_ar1", "searev", "coarse_controls", "uww",
                                   "storage_ar1_w2", "storage_ar1_w4", "storage_ar1_w7"])
def test_hoisted_inner_interpolation_is_bit_identical(product, which):
    """AF kernel with and without the per-item table of inner interpolations; the
    constant-W kernel with all slots live (W = 3, 5, 9) and with idle slots (W = 2, 4, 7)"""
    import workloads as wl
    from stodynprog_b200 import _cabi
    api = _Api(product, "cuda", "control_minor", "auto", "on")
    if which.startswith("storage_ar1_w"):
        sv = wl.storage_ar1(api, n_E=9, n_P=11, n_w=int(which[-1]), steps=(0.01, 0.1)).solver
    else:
        sv = _factor_case(api, which)
    assert sv.sweep_tables().u_mask == 1
    lib = sv.engine.lib
    J0 = np.random.default_rng(3).standard_normal(sv._state_grid_shape)
    J0[0] = np.nan if which == "uww" else J0[0]
    out = {}
    try:
        # hoist_const = 1: the constant-W kernel (W <= 9, the default); 0: the runtime-W kernel
        for hoist, const in ((1, 1), (1, 0), (0, 0)):
            for upl in (4, 2):
                _cabi.check(lib.sdp_set_option(b"hoist", hoist), "sdp_set_option")
                _cabi.check(lib.sdp_set_option(b"hoist_const", const), "sdp_set_option")
                _cabi.check(lib.sdp_set_option(b"upl", upl), "sdp_set_option")
                _cabi.check(lib.sdp_set_option(b"hoist_upl", upl), "sdp_set_option")
                out[hoist, const, upl] = sv.value_iteration(J0, report_time=False)
    finally:
        lib.sdp_set_option(b"hoist", 1)
        lib.sdp_set_option(b"hoist_const", 1)
        lib.sdp_set_option(b"upl", 4)
        lib.sdp_set_option(b"hoist_upl", 2)
    Jr, polr = out[0, 0, 4]
    for key, (J, pol) in out.items():
        assert np.array_equal(J.view(np.int64), Jr.view(np.int64)), key
        assert np.array_equal(pol, polr, equal_nan=True), key


# ---------------------------------------------------------------------------
# layout CF (column-shared hoist): BF tables over column-major tiles, one inner-
# interpolation table per column of the grid - bit-identical to layout BF
# ---------------------------------------------------------------------------
def _coupled_w_system(api, n0=40, **kw):
    """u_mask == 1, but the perturbed coordinate also depends on state axis 0: the
    (x,w) part varies along a column, so layout CF must be refused"""
    import scipy.stats as stats

    def dyn(x0, x1, u, w):
        return (0.9 * x0 + 0.5 * u, 0.7 * x1 + 0.05 * x0 + w)

    def box(x0, x1):
        return ((-1.0, 1.0 + 0.1 * x0),)

    def cost(x0, x1, u, w):
        return x0 ** 2 + x1 ** 2 + 0.1 * u ** 2

    sys = api.SysDescription((2, 1, 1), name='coupled w')
    sys.dyn, sys.control_box, sys.cost = dyn, box, cost
    sys.perturb_laws = [stats.norm(0, 0.3)]
    sv = api.DPSolver(sys, **kw)
    sv.discretize_state(-1.0, 2.0, n0, -1.0, 1.0, 5)
    sv.discretize_perturb(-0.9, 0.9, 5)
    sv.control_steps = (0.25,)
    return sv


def _column_case(api, which):
    import workloads as wl
    if which.startswith("ar1_w"):
        # 70 rows: 3 tiles per column, the last one with 26 padding lanes; control step 0.5 =
        # 3.5 grid rows; W = 9, 5, 3 fill the unrolled slots, W = 7, 4, 2 leave idle ones
        return wl.storage_ar1(api, n_E=70, n_P=5, n_w=int(which[5:]), steps=(0.5, 0.1)).solver
    if which == "ar1_exact_tiles":
        return wl.storage_ar1(api, n_E=64, n_P=3, n_w=3, steps=(0.25, 0.1)).solver
    if which == "searev":                       # d = 3: a column is a (speed, acceleration) pair
        prob = wl.searev(api, n_E=33, n_S=4, n_A=3)
        prob.solver.control_steps = (.05,)
        return prob.solver
    if which == "curtail":                      # two controls, ragged in both axes
        sv = _two_control_system(api)
        sv.discretize_state(0, 10., 35, -4, 4, 4)
        return sv
    raise KeyError(which)


COLUMN_CASES = ["ar1_w9", "ar1_w7", "ar1_w5", "ar1_w4", "ar1_w3", "ar1_w2", "ar1_exact_tiles",
                "searev", "curtail"]


def _same_bits(a, b):
    """bit-identical, except that any NaN matches any NaN: which of two NaN operands (or
    which sign of a generated NaN) an fp64 instruction returns depends on the operand order
    the compiler picked for a commutative operation, not on the algorithm - and numpy's
    argmin (stodynprog.py:686) does not tell NaNs apart either"""
    a, b = np.asarray(a), np.asarray(b)
    na, nb = np.isnan(a), np.isnan(b)
    return bool(np.array_equal(na, nb) and np.array_equal(a[~na].view(np.int64), b[~nb].view(np.int64)))


@pytest.mark.parametrize("backend", [pytest.param("model"), pytest.param("cuda", marks=gpu)])
@pytest.mark.parametrize("which", COLUMN_CASES)
def test_column_hoist_is_bit_identical(product, backend, which):
    """layout CF against layout BF (same factored entries, states walked column by column,
    the inner interpolation tabulated once per column): J and policies bit for bit, NaN
    and infinities in J included; item chunking does not matter"""
    if backend == "model" and which in ("ar1_w7", "ar1_w5", "ar1_w4", "ar1_w2"):
        pytest.skip("the numpy model does not depend on W; covered on the GPU")
    ref = _column_case(_Api(product, backend, "state_minor", "auto", "on"), which)
    ref.column_hoist = "off"
    col = _column_case(_Api(product, backend, "state_minor", "auto", "on"), which)
    col.column_hoist, col.column_pairs = "on", "off"        # one row per lane
    col2 = _column_case(_Api(product, backend, "state_minor", "auto", "on"), which)
    col2.column_hoist, col2.column_pairs = "on", "on"       # two rows per lane
    J0 = np.random.default_rng(11).standard_normal(ref._state_grid_shape)
    for sweep in range(3):
        Jr, polr = ref.value_iteration(J0, report_time=False)
        Jc, polc = col.value_iteration(J0, report_time=False)
        Jc2, polc2 = col2.value_iteration(J0, report_time=False)
        Tr, Tc, Tc2 = ref.last_tables, col.last_tables, col2.last_tables
        assert Tr.layout_name == "state_minor_factored" and Tc.layout_name == "column_factored"
        assert Tc2.layout_name == "column_factored" and Tc2.pairs and not Tc.pairs
        assert Tc.n_backups_local == Tr.n_backups_local == Tc2.n_backups_local and Tc.u_mask == 1
        assert _same_bits(Jr, Jc) and _same_bits(Jr, Jc2), sweep
        assert np.array_equal(polr, polc, equal_nan=True) and np.array_equal(polr, polc2, equal_nan=True), sweep
        J0 = Jr.copy()
        if sweep == 1:                          # special values travel through the table too
            J0.reshape(-1)[::7] = np.nan
            J0.reshape(-1)[3::11] = np.inf
    if backend == "cuda":
        # CTA size, controls per iteration and work-item length do not change a bit
        lib = col.engine.lib
        try:
            Jr, polr = ref.value_iteration(J0, report_time=False)
            for threads, ub, pf, pre in ((128, 1, 1, 1), (256, 2, 1, 0), (512, 1, 2, 0), (96, 2, 2, 2),
                                         (160, 1, 2, 1), (640, 2, 1, 2), (640, 2, 2, 1), (768, 2, 1, 2),
                                         (768, 1, 2, 0), (704, 1, 1, 2), (768, 2, 1, 3), (640, 1, 2, 3),
                                         (64, 2, 2, 3)):
                lib.sdp_set_option(b"col_threads", threads)
                lib.sdp_set_option(b"col_ub", ub)
                lib.sdp_set_option(b"col_pf", pf)
                lib.sdp_set_option(b"col_prepass", pre)
                lib.sdp_set_option(b"col_dynamic", (threads // 32) % 2)
                J2, pol2 = col.value_iteration(J0, report_time=False)
                assert _same_bits(Jr, J2), (threads, ub, pf, pre)
                assert np.array_equal(polr, pol2, equal_nan=True), (threads, ub, pf, pre)
                if pre >= 2:            # (two rows per lane copies its table with the TMA engine only)
                    J3, pol3 = col2.value_iteration(J0, report_time=False)
                    assert _same_bits(Jr, J3) and np.array_equal(polr, pol3, equal_nan=True), (threads, "pairs")
        finally:
            lib.sdp_set_option(b"col_threads", 768)
            lib.sdp_set_option(b"col_ub", 2)
            lib.sdp_set_option(b"col_pf", 2)
            lib.sdp_set_option(b"col_prepass", 3)
            lib.sdp_set_option(b"col_dynamic", 1)


@pytest.mark.parametrize("backend", [pytest.param("model"), pytest.param("cuda", marks=gpu)])
def test_column_hoist_solvers_and_chunking(product, backend):
    """the other drivers on top of layout CF: relative DP, policy iteration, the
    device-resident loop; explicit work-item lengths"""
    import workloads as wl
    out = []
    for colmode, chunk in (("off", None), ("on", None), ("on", 4), ("on", 512)):
        api = _Api(product, backend, "state_minor", "auto", "on")
        prob = wl.storage_ar1(api, n_E=40, n_P=4, n_w=5, steps=(0.5, 0.1), item_chunk=chunk)
        sv = prob.solver
        sv.column_hoist = colmode
        J0 = np.random.default_rng(2).standard_normal(sv._state_grid_shape)
        J0[sv._state_ref_ind] = 0.
        (Jd, Jref), pol = sv.value_iteration((J0, 0.), rel_dp=True, report_time=False)
        assert sv.last_tables.column == (colmode == "on")
        (Jp, Jpr), polp = sv.policy_iteration(prob.initial_policy(), 5, 2, rel_dp=True)
        Js, pols, info = sv.solve_value_iteration(J_zero=J0, max_iter=3, tol=0.0)
        out.append((Jd, Jref, pol, Jp, Jpr, polp, Js, pols, np.array(info["residuals"])))
    for other in out[1:]:
        for a, b in zip(out[0], other):
            assert np.array_equal(np.asarray(a).view(np.int64), np.asarray(b).view(np.int64))


@pytest.mark.parametrize("backend", [pytest.param("model"), pytest.param("cuda", marks=gpu)])
@pytest.mark.parametrize("colmode", ["on", "off"])
def test_column_cases_golden(product, backend, colmode, capsys):
    """fixtures generated from the unmodified reference on grids that layout CF takes
    (tests/golden/column_cases.npz): value iteration from 0 and from a random J, policy
    iteration with relative DP (2-D storage-AR1, 70 x 5) and value iteration on a 3-D SEAREV
    grid (33 x 4 x 3) - through layout CF and, for comparison, through layout BF"""
    from golden_cases import column_cases
    G = golden("column_cases.npz")
    ar1, sea = column_cases(_Api(product, backend, "state_minor", "auto", "on", colmode))
    want_layout = "column_factored" if colmode == "on" else "state_minor_factored"
    J = ar1.J0
    for k in range(3):
        J, pol = ar1.solver.value_iteration(J, report_time=False)
        assert ar1.solver.last_tables.layout_name == want_layout
        n_bad, _ = policy_mismatch_report(pol, G["ar1_vi_pol%d" % k])
        assert n_bad == 0 and rel_err(J, G["ar1_vi_J%d" % k]) <= J_RTOL, k
    J, pol = ar1.solver.value_iteration(G["ar1_J_rand"], report_time=False)
    n_bad, _ = policy_mismatch_report(pol, G["ar1_vr_pol"])
    assert n_bad == 0 and rel_err(J, G["ar1_vr_J"]) <= J_RTOL
    (Jd, Jr), pol = ar1.solver.policy_iteration(ar1.initial_policy(), 10, 2, rel_dp=True)
    n_bad, _ = policy_mismatch_report(pol, G["ar1_pi_pol"])
    assert n_bad == 0 and abs(Jr - float(G["ar1_pi_Jref"])) <= J_RTOL * abs(float(G["ar1_pi_Jref"]))
    assert np.max(np.abs(Jd - G["ar1_pi_J"])) <= J_RTOL * np.max(np.abs(G["ar1_pi_J"]))
    printed = [float(l.split(':')[1]) for l in capsys.readouterr().out.splitlines() if 'ref policy cost' in l]
    assert ['{:g}'.format(c) for c in printed] == ['{:g}'.format(c) for c in G["ar1_pi_ref_costs"]]
    J = sea.J0
    for k in range(2):
        J, pol = sea.solver.value_iteration(J, report_time=False)
        assert sea.solver.last_tables.layout_name == want_layout
        n_bad, _ = policy_mismatch_report(pol, G["sea_vi_pol%d" % k])
        assert n_bad == 0 and rel_err(J, G["sea_vi_J%d" % k]) <= J_RTOL, k


@pytest.mark.parametrize("backend", [pytest.param("model"), pytest.param("cuda", marks=gpu)])
@pytest.mark.parametrize("which", ["ar1_w3_tall", "searev_tall"])
def test_column_hoist_row_bands(product, backend, which, monkeypatch):
    """layout CF with the rows cut into several bands (tiles ordered band by band, one
    combine launch per band): same J and policies, bit for bit, as one band and as BF"""
    import workloads as wl
    from stodynprog_b200.engine import Engine
    out = {}
    for bands in ("off", "1", "3", "5"):
        monkeypatch.setattr(Engine, "COLUMN_BANDS", "1" if bands == "off" else bands)
        api = _Api(product, backend, "state_minor", "auto", "on")
        if which == "ar1_w3_tall":
            sv = wl.storage_ar1(api, n_E=330, n_P=3, n_w=3, steps=(2.0, 0.1)).solver
        else:
            prob = wl.searev(api, n_E=330, n_S=3, n_A=2)
            prob.solver.control_steps = (.2,)
            sv = prob.solver
        sv.column_hoist = "off" if bands == "off" else "on"
        J0 = np.random.default_rng(8).standard_normal(sv._state_grid_shape)
        J1, pol1 = sv.value_iteration(J0, report_time=False)
        T = sv.last_tables
        if bands != "off":
            assert T.column and len(T.bands["tiles"]) == int(bands)
            assert T.bands["rows"][0] == 0 and T.bands["rows"][-1] == sv._state_grid_shape[0]
            assert all(r % 32 == 0 for r in T.bands["rows"][:-1])
        J2, pol2 = sv.value_iteration(J1, report_time=False)
        out[bands] = (J1, pol1, J2, pol2)
    for bands, res in out.items():
        for a, b in zip(out["off"], res):
            assert np.array_equal(a.view(np.int64), b.view(np.int64)), bands


def test_column_hoist_band_launch_plan(product, monkeypatch):
    """the launch sequence of value_iteration's large-sweep path for layout CF, replayed on
    the numpy model: pre-pass once, then per row band one streaming launch over the band's
    own CTA segments (col_table_ready = 1) and one combine launch on the band's view - the
    union must equal the one-launch sweep"""
    import ctypes
    import torch
    import workloads as wl
    from stodynprog_b200.engine import Engine
    monkeypatch.setattr(Engine, "COLUMN_BANDS", "3")
    api = _Api(product, "model", "state_minor", "auto", "on")
    sv = wl.storage_ar1(api, n_E=330, n_P=3, n_w=3, steps=(2.0, 0.1)).solver
    sv.column_hoist = "on"
    T = sv.sweep_tables()
    eng = sv.engine
    assert T.column and len(T.bands["tiles"]) == 3 and not eng.can_overlap_results(T)   # (no GPU here)
    n_grid = 330 * 3
    J = torch.from_numpy(np.random.default_rng(3).standard_normal(n_grid))
    J_ref = torch.empty(n_grid, dtype=torch.float64)
    eng.sweep(T, J, J_ref)
    argmin_ref = T.argmin[:n_grid].clone()
    plan = eng._chunk_plan(T)
    assert len(plan) == 3 and plan is eng._chunk_plan(T)
    assert [ch["s0"] for ch in plan] == [r * 3 for r in T.bands["rows"][:-1]]
    assert [ch["s1"] for ch in plan] == [r * 3 for r in T.bands["rows"][1:]]
    T.part_val.fill_(float("nan"))
    T.argmin.fill_(-7)
    J_new = torch.full((n_grid,), float("nan"), dtype=torch.float64)
    lib = eng.lib
    assert lib.sdp_column_table(ctypes.byref(T.grid), ctypes.byref(T.c_tables), eng._ptr(J), eng.stream) == 0
    tb0 = T.bands["tile_begin"]
    for b, ch in enumerate(plan):
        seg = ch["keep"].numpy()
        # (positions of the work list: every item, or - two rows per lane - the first tile's of each pair)
        i0, i1 = (int(np.searchsorted(T.work_host, T.item_begin_host[tb0[k]])) for k in (b, b + 1))
        assert seg[0] == i0 and seg[-1] == i1 and np.all(np.diff(seg) >= 0) and i1 > i0
        assert ch["tab_p"].col_table_ready == 1 and ch["tab_p"].n_segs == len(seg) - 1
        assert ch["tab_f"].n_states == ch["s1"] - ch["s0"] and ch["tab_f"].tiles_per_col == T.bands["tiles"][b]
        assert lib.sdp_sweep_partials(ctypes.byref(T.grid), ctypes.byref(ch["tab_p"]), eng._ptr(J), ch["pv"],
                                      ch["pi"], eng.stream) == 0
        assert lib.sdp_sweep_finalize(ctypes.byref(ch["tab_f"]), eng._ptr(T.part_val), eng._ptr(T.part_idx),
                                      ctypes.c_void_p(J_new.data_ptr() + 8 * ch["s0"]),
                                      ctypes.c_void_p(T.argmin.data_ptr() + 4 * ch["s0"]), eng.stream) == 0
    assert torch.equal(J_new.view(torch.int64), J_ref.view(torch.int64))
    assert torch.equal(T.argmin[:n_grid], argmin_ref)
    # re-cutting the CTA segments invalidates the cached plan and band views
    eng.set_column_segments(T, 7)
    assert T.n_segs == 7 and T.chunk_plan is None and T.band_views is None
    J_again = torch.empty(n_grid, dtype=torch.float64)
    eng.sweep(T, J, J_again)
    assert torch.equal(J_again.view(torch.int64), J_ref.view(torch.int64))


def test_column_piece_launch_plan(product, monkeypatch):
    """the launch sequence of value_iteration's large-sweep path for layout CF with one band,
    replayed on the numpy model: pre-pass once, then per PIECE OF COLUMNS one streaming launch over
    the piece's own CTA segments, one combine launch on the piece's view that also maps the argmin
    to control values, and 2-D copies of the piece's columns into the C-order result arrays - the
    union must equal the one-launch sweep followed by sdp_policy_values"""
    import ctypes
    import torch
    import workloads as wl
    from stodynprog_b200.engine import Engine
    monkeypatch.setattr(Engine, "COLUMN_PIECES", (0.4, 0.3, 0.2, 0.1))
    api = _Api(product, "model", "state_minor", "auto", "on")
    sv = wl.storage_ar1(api, n_E=70, n_P=11, n_w=3, steps=(1.0, 0.1)).solver
    sv.column_hoist = "on"
    T = sv.sweep_tables()
    eng = sv.engine
    n_rows, n_cols, nc = 70, 11, 2
    n_grid = n_rows * n_cols
    assert T.column and len(T.bands["tiles"]) == 1 and T.n_cols == n_cols
    J = torch.from_numpy(np.random.default_rng(3).standard_normal(n_grid))
    J_ref = torch.empty(n_grid, dtype=torch.float64)
    eng.sweep(T, J, J_ref)
    argmin_ref = T.argmin[:n_grid].clone()
    pol_ref = eng.policy_values(T, argmin_ref)
    plan = eng._chunk_plan(T)
    assert plan is eng._chunk_plan(T) and len(plan) == 4
    assert [ch["c0"] for ch in plan][0] == 0 and [ch["c1"] for ch in plan][-1] == n_cols
    assert all(a["c1"] == b["c0"] and a["c0"] < a["c1"] for a, b in zip(plan, plan[1:]))
    widths = [ch["c1"] - ch["c0"] for ch in plan]
    assert widths[0] == max(widths) and sum(widths) == n_cols
    T.part_val.fill_(float("nan"))
    T.argmin.fill_(-7)
    J_new = torch.full((n_grid,), float("nan"), dtype=torch.float64)
    pol = torch.full((n_grid, nc), float("nan"), dtype=torch.float64)
    J_host = torch.full((n_grid,), float("nan"), dtype=torch.float64)
    pol_host = torch.full((n_grid, nc), float("nan"), dtype=torch.float64)
    eng._copy = type("S", (), {"cuda_stream": 0})()
    lib = eng.lib
    assert lib.sdp_column_table(ctypes.byref(T.grid), ctypes.byref(T.c_tables), eng._ptr(J), eng.stream) == 0
    tpc = T.bands["tiles"][0]
    for ch in plan:
        seg = ch["keep"].numpy()
        i0, i1 = (int(T.item_begin_host[c * tpc]) for c in (ch["c0"], ch["c1"]))
        assert seg[0] == i0 and seg[-1] == i1 and np.all(np.diff(seg) >= 0) and i1 > i0
        assert ch["tab_p"].col_table_ready == 1 and ch["tab_p"].n_segs == len(seg) - 1
        assert ch["tab_f"].n_cols == ch["c1"] - ch["c0"] and ch["tab_f"].n_states == n_rows * ch["tab_f"].n_cols
        assert lib.sdp_sweep_partials(ctypes.byref(T.grid), ctypes.byref(ch["tab_p"]), eng._ptr(J), ch["pv"],
                                      ch["pi"], eng.stream) == 0
        assert lib.sdp_sweep_finalize_cols(
            ctypes.byref(ch["tab_f"]), eng._ptr(T.part_val), eng._ptr(T.part_idx), eng._ptr(J_new),
            eng._ptr(T.argmin), n_cols, ch["c0"], nc, eng._ptr(T.lo_dev), eng._ptr(T.hi_dev),
            eng._ptr(T.npts_dev), eng._ptr(pol), int(ch is not plan[-1]), eng.stream) == 0
        eng._columns_to_host(T, ch, J_new, pol, J_host, pol_host)
    for got in (J_new, J_host):
        assert torch.equal(got.view(torch.int64), J_ref.view(torch.int64))
    for got in (pol, pol_host):
        assert torch.equal(got.view(torch.int64), pol_ref.reshape(n_grid, nc).view(torch.int64))
    assert torch.equal(T.argmin[:n_grid], argmin_ref)
    # fewer columns than pieces: as many pieces as there are columns to cut
    sv2 = wl.storage_ar1(api, n_E=40, n_P=2, n_w=3, steps=(1.0, 0.1)).solver
    sv2.column_hoist = "on"
    T2 = sv2.sweep_tables()
    p2 = sv2.engine._chunk_plan(T2)
    assert [(ch["c0"], ch["c1"]) for ch in p2] == [(0, 1), (1, 2)]


def test_column_bands_choice(product, monkeypatch):
    """row bands of layout CF: none on several ranks or small slabs, whole tiles of 32 rows,
    cut by the controls of the rows"""
    from stodynprog_b200.engine import Engine
    from fake_lib import FakeLib
    eng = Engine(_test_lib=FakeLib())
    w = np.full(2000, 205.0)
    monkeypatch.setattr(Engine, "COLUMN_BANDS", "1")
    assert eng._column_bands(w, 9) == [0, 2000]
    monkeypatch.setattr(Engine, "COLUMN_BANDS", "auto")
    assert eng._column_bands(w, 9) == [0, 2000]            # results leave by pieces of columns
    monkeypatch.setattr(Engine, "COLUMN_BANDS", "3")
    assert eng._column_bands(w, 9) == [0, 928, 1408, 2000]
    assert eng._column_bands(np.r_[np.full(1000, 100.0), np.full(1000, 300.0)], 9) == [0, 1280, 1600, 2000]
    monkeypatch.setattr(Engine, "COLUMN_BANDS", "5")
    b = eng._column_bands(w, 9)
    assert len(b) == 6 and all(x % 32 == 0 for x in b[:-1]) and b[-1] == 2000
    assert eng._column_bands(np.full(100, 205.0), 9) == [0, 100]      # too few rows for 5 bands
    eng.coll.world = 2
    assert eng._column_bands(w, 9) == [0, 2000]            # one epoch per sweep and rank


def test_column_hoist_is_refused_when_it_does_not_apply(product):
    """a w-part that varies along a column is detected on the built tables: "auto" falls
    back to layout BF (same results), "on" raises; so do grids or layouts CF cannot take"""
    import stodynprog_b200.tablebuild as engine_mod
    ref = _coupled_w_system(_Api(product, "model", "state_minor", "auto", "on"))
    ref.column_hoist = "off"
    auto = _coupled_w_system(_Api(product, "model", "state_minor", "auto", "on"))
    saved = engine_mod.COLUMN_HOIST_DEFAULT
    engine_mod.COLUMN_HOIST_DEFAULT = True
    try:
        J0 = np.random.default_rng(4).standard_normal(ref._state_grid_shape)
        Jr, polr = ref.value_iteration(J0, report_time=False)
        Ja, pola = auto.value_iteration(J0, report_time=False)
        assert auto.last_tables.layout_name == "state_minor_factored"     # refused, rebuilt as BF
        assert np.array_equal(Jr.view(np.int64), Ja.view(np.int64)) and np.array_equal(polr, pola)
        # ... and "auto" takes it when it applies
        ok = _column_case(_Api(product, "model", "state_minor", "auto", "on"), "ar1_exact_tiles")
        assert ok.sweep_tables().layout_name == "column_factored"
    finally:
        engine_mod.COLUMN_HOIST_DEFAULT = saved
    forced = _coupled_w_system(_Api(product, "model", "state_minor", "auto", "on"))
    forced.column_hoist = "on"
    with pytest.raises(ValueError):
        forced.sweep_tables()
    few_rows = _coupled_w_system(_Api(product, "model", "state_minor", "auto", "on"), n0=20)
    few_rows.column_hoist = "on"
    with pytest.raises(ValueError):
        few_rows.sweep_tables()
    wrong_layout = _column_case(_Api(product, "model", "control_minor", "auto", "on"), "ar1_exact_tiles")
    wrong_layout.column_hoist = "on"
    with pytest.raises(ValueError):
        wrong_layout.sweep_tables()
    bad = _column_case(_Api(product, "model", "state_minor", "auto", "on"), "ar1_exact_tiles")
    bad.column_hoist = "sometimes"
    with pytest.raises(ValueError):
        bad.sweep_tables()


def test_unfactorable_systems_fall_back_to_dense(product):
    """a coordinate that spans controls AND perturbation, or a cost that depends
    on w, keeps the dense tables in "auto" mode and is refused in "on" mode"""
    for kind in ("plain", "w"):
        sv = _toy(_Api(product, "model", "control_minor", "auto", "auto"), 2, kind)
        assert not sv.sweep_tables().factored
    sv = _toy(_Api(product, "model", "control_minor", "auto", "on"), 2)
    with pytest.raises(ValueError):
        sv.sweep_tables()
    # deterministic and 1-D systems have nothing to factor
    import workloads as wl
    api = _Api(product, "model", "control_minor", "auto", "auto")
    assert not wl.inventory(api).solver.sweep_tables().factored


def _two_control_system(api, **kw):
    """storage + AR(1) with curtailment enabled: the second control's grid
    depends on the state (U2 = [0, max(P_mis, 0)]), so the control product is
    ragged in both axes (notebook cell 5 with curt_activ = True)."""
    import scipy.stats as stats
    E_rated, P_rated, p_corr = 10., 4., 0.8

    def dyn_sto(E, P_mis, P_sto, P_cur, innov):
        return (E + P_sto, p_corr * P_mis + innov)

    def admissible_controls(E, P_mis):
        return ((np.max((-E, -P_rated)), np.min((E_rated - E, P_rated))), (0, np.max((P_mis, 0))))

    def cost(E, P_mis, P_sto, P_cur, innov):
        P_dev = P_mis - P_cur - P_sto
        return P_dev ** 2 + 0.3 * P_cur

    sys = api.SysDescription((2, 2, 1), name='storage with curtailment')
    sys.dyn = dyn_sto
    sys.control_box = admissible_controls
    sys.cost = cost
    sys.perturb_laws = [stats.norm(0, 0.4)]
    sv = api.DPSolver(sys, **kw)
    sv.discretize_state(0, E_rated, 7, -4, 4, 9)
    sv.discretize_perturb(-1.2, 1.2, 5)
    sv.control_steps = (0.5, 0.25)
    return sv


def test_two_controls_ragged_product(api, port):
    sv, so = _two_control_system(api), _two_control_system(port)
    J0 = np.random.default_rng(11).standard_normal(sv._state_grid_shape)
    J, pol = sv.value_iteration(J0, report_time=False)
    Jo, polo = so.value_iteration(J0)
    assert sv.last_tables.host_full.npts[:, 1].min() == 1
    assert sv.last_tables.host_full.npts[:, 1].max() > 5
    assert np.array_equal(pol, polo)
    assert rel_err(J, Jo) <= J_RTOL


# ---------------------------------------------------------------------------
# config #4 at full size: the reference's shipped golden policy
# ---------------------------------------------------------------------------
@gpu
def test_searev_full_policy_iteration_golden(cuda_api, capsys):
    """examples/20 .../storage control/pol_E10_grid3161_iter5.npy: the policy after
    policy_iteration(pol_lin, 1000, 5, rel_dp=True) on the 31x61x61 grid (5 argmin
    sweeps over 2.2 G backups + 6000 fixed-policy backups of the whole grid).  The
    fixture is the unmodified reference's output, bit-identical to the shipped file."""
    import workloads as wl
    G = golden("searev_full.npz")
    assert bool(G["matches_shipped_npy"])
    prob = wl.searev(cuda_api)
    (Jd, Jr), pol = prob.solver.policy_iteration(prob.initial_policy(), 1000, 5, rel_dp=True)
    text = capsys.readouterr().out
    costs = [l.split(':')[1].strip() for l in text.splitlines() if 'ref policy cost' in l]
    assert costs == ['{:g}'.format(c) for c in G["pi_ref_costs"]]
    assert costs == ['0.0864223', '0.0798338', '0.0760902', '0.0747645', '0.0746698', '0.0746743']
    assert prob.solver.last_tables.n_backups_total == 2211312159
    n_bad, diff = policy_mismatch_report(pol, G["pi_pol"])
    # exact agreement is expected; a handful of near-ties (two controls whose
    # expected costs differ by a few ulp) would be reported here, not hidden
    print("SEAREV golden policy: %d / %d states differ" % (n_bad, diff.size))
    assert n_bad == 0
    assert abs(Jr - float(G["pi_Jref"])) <= J_RTOL * abs(float(G["pi_Jref"]))
    assert np.max(np.abs(Jd - G["pi_J"])) <= J_RTOL * np.max(np.abs(G["pi_J"]))


@gpu
def test_sharded_two_gpus_subprocess():
    """N > 1 on real GPUs (skipped on a 1-GPU box): tests/multi_gpu_check.py"""
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import os
    from conftest import ROOT
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", "29517",
           os.path.join(ROOT, "tests", "multi_gpu_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "MULTI_GPU_PARITY OK" in res.stdout


# ---------------------------------------------------------------------------
# full-size properties (config #5 is too big for the CPU oracle: sampled check)
# ---------------------------------------------------------------------------
@gpu
def test_large_grid_sampled_against_port(cuda_api, port):
    """2000 x 125 slice of config #5 (layout B, batched tabulation): 300 random
    states checked against the numpy port; min over controls <= any fixed control;
    idempotence of the table cache."""
    import workloads as wl
    n_E, n_P = 2000, 125
    prob = wl.storage_ar1_large(cuda_api, n_E=n_E, n_P=n_P)
    ora = wl.storage_ar1_large(port, n_E=n_E, n_P=n_P)
    sv = prob.solver
    J0 = np.random.default_rng(0).standard_normal((n_E, n_P))
    J, pol = sv.value_iteration(J0, report_time=False)
    T = sv.last_tables
    assert T.tiled and T.tabulate_mode == "batched"
    J2, pol2 = sv.value_iteration(J0, report_time=False)
    assert sv.last_tables is T and np.array_equal(J, J2) and np.array_equal(pol, pol2)
    Ji = ora.solver.interp_on_state(J0)
    rng = np.random.default_rng(1)
    for flat in rng.choice(n_E * n_P, size=300, replace=False):
        idx = np.unravel_index(flat, (n_E, n_P))
        x_k = tuple(g[i] for g, i in zip(ora.solver.state_grid, idx))
        Jo, uo = ora.solver.value_at_state(x_k, Ji)
        assert list(pol[idx]) == list(uo)
        assert abs(J[idx] - Jo) <= J_RTOL * max(abs(Jo), 1e-300)
    # the greedy value never exceeds the value of the 'do nothing'-like first control
    Je = sv.eval_policy(pol, 1, J_zero=J0, report_time=False)
    assert np.max(np.abs(Je - J)) <= 1e-10 * np.max(np.abs(J))


@gpu
def test_device_argument_is_honoured(product, port):
    """DPSolver(sys, device='cuda:1') while device 0 is current: buffers AND launches go to
    GPU 1 (the C ABI launches on the current device, so the engine makes its device current
    around every entry point); the caller's current device is left alone"""
    import torch
    import workloads as wl
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    torch.cuda.set_device(0)
    kw = dict(n_E=9, n_P=11, steps=(0.01, 0.1))
    sv = wl.storage_ar1(product, device="cuda:1", **kw).solver
    ora = wl.storage_ar1(port, **kw).solver
    J = np.random.default_rng(0).standard_normal((9, 11))
    for _ in range(2):
        Jg, polg = sv.value_iteration(J, report_time=False)
        Jo, polo = ora.value_iteration(J)
        assert policy_mismatch_report(polg, polo)[0] == 0 and rel_err(Jg, Jo) <= J_RTOL
        J = Jo
    assert sv.last_tables.cell.device.index == 1 and torch.cuda.current_device() == 0
    pol0 = wl.storage_ar1(product, **kw).initial_policy()
    assert rel_err(sv.eval_policy(pol0, 5, report_time=False), ora.eval_policy(pol0, 5)) <= J_RTOL


@gpu
def test_config5_full_size_against_port(cuda_api, port):
    """BASELINE configs[4] at FULL size - 2000 x 500 states x 129..256 controls x 9 nodes,
    1 848 240 000 backups per sweep - through the default tables (layout CF, one band):
    `value_iteration` (results streamed by pieces of columns, Engine.sweep_to_host) and the
    device-resident loop (Engine.sweep), 1 000 seeded random states against the oracle port
    (stodynprog.py:639-691): policies exact, J within 1e-10."""
    import workloads as wl
    prob = wl.storage_ar1_large(cuda_api)
    ora = wl.storage_ar1_large(port).solver
    sv = prob.solver
    dims = sv._state_grid_shape
    assert dims == (2000, 500)
    J0 = np.random.default_rng(3).standard_normal(dims)
    J, pol = sv.value_iteration(J0, report_time=False)
    T = sv.last_tables
    assert T.layout_name == "column_factored" and len(T.bands["tiles"]) == 1
    assert sv.engine.can_overlap_results(T) and len(sv.engine._chunk_plan(T)) == 4
    assert T.n_backups_total == 1848240000
    Js, pols, info = sv.solve_value_iteration(J_zero=J0, max_iter=1)
    assert np.array_equal(J.view(np.int64), Js.view(np.int64)) and np.array_equal(pol, pols)
    Ji = ora.interp_on_state(J0)
    n_bad, worst = 0, 0.0
    for flat in np.random.default_rng(4).choice(J0.size, size=1000, replace=False):
        idx = np.unravel_index(flat, dims)
        x_k = tuple(g[i] for g, i in zip(ora.state_grid, idx))
        Jo, uo = ora.value_at_state(x_k, Ji)
        n_bad += list(pol[idx]) != list(uo)
        worst = max(worst, abs(J[idx] - Jo) / max(abs(Jo), 1e-300))
    assert n_bad == 0 and worst <= J_RTOL, (n_bad, worst)


@gpu
@pytest.mark.parametrize("n_w", [3, 4, 5, 9])
def test_column_layout_against_port_by_W(cuda_api, port, n_w):
    """layout CF against the oracle port on every state, for the node counts that take the
    3-, 5- and 9-slot instantiations of the column kernel exactly (FULL) and partly (W = 4:
    slot masking)"""
    import workloads as wl
    kw = dict(n_E=70, n_P=6, n_w=n_w, steps=(0.3, 0.1))
    sv = wl.storage_ar1(cuda_api, **kw).solver
    sv.table_layout, sv.column_hoist = "state_minor", "on"
    ora = wl.storage_ar1(port, **kw).solver
    J = np.random.default_rng(n_w).standard_normal((70, 6))
    for sweep in range(2):
        Jg, polg = sv.value_iteration(J, report_time=False)
        assert sv.last_tables.layout_name == "column_factored"
        Jo, polo = ora.value_iteration(J)
        assert policy_mismatch_report(polg, polo)[0] == 0
        assert rel_err(Jg, Jo) <= J_RTOL
        J = Jo


@gpu
def test_layout_B_kernel_variants_are_bit_identical(product):
    """straight LDG, TMA-fed ring (several ring shapes) and software-pipelined
    kernels of the state-minor layout, and both lane widths of layout A, must
    produce identical J and argmin"""
    import workloads as wl
    from stodynprog_b200 import _cabi
    lib = _cabi.load_library()

    def opt(**kw):
        for k, v in kw.items():
            _cabi.check(lib.sdp_set_option(k.encode(), int(v)), "sdp_set_option")
    try:
        for layout, settings in (
                ("state_minor", [dict(tma=0, wb=1), dict(tma=0, wb=3), dict(tma=2, rb=2), dict(tma=2, rb=4),
                                 dict(tma=2, rb=8), dict(tma=1, tma_rows=8, tma_stages=2, tma_warps=4),
                                 dict(tma=1, tma_rows=4, tma_stages=3, tma_warps=8),
                                 dict(tma=1, tma_rows=8, tma_stages=5, tma_warps=2)]),
                ("control_minor", [dict(upl=4), dict(upl=2)])):
            for which in ("ar1", "toy3w", "searev"):
                api = _Api(product, "cuda", layout)
                if which == "ar1":
                    sv = wl.storage_ar1(api, n_E=40, n_P=37, steps=(0.05, 0.1), item_chunk=48).solver
                elif which == "toy3w":
                    sv = _toy(api, 3, "w", item_chunk=8)
                else:
                    sv = _searev_small(api).solver
                J0 = np.random.default_rng(4).standard_normal(sv._state_grid_shape)
                ref = None
                for st in settings:
                    opt(**st)
                    J, pol = sv.value_iteration(J0, report_time=False)
                    if ref is None:
                        ref = (J, pol)
                    assert np.array_equal(J, ref[0]) and np.array_equal(pol, ref[1]), (layout, which, st)
    finally:
        opt(tma=1, tma_rows=8, tma_stages=2, tma_warps=4, rb=4, wb=1, upl=4)


@gpu
@pytest.mark.parametrize("layout", ["control_minor", "state_minor"])
@pytest.mark.parametrize("compress", ["off", "auto"])
def test_overlapped_result_copy_is_bit_identical(product, layout, compress):
    """value_iteration's large-sweep path (runs of the slab swept on alternating streams,
    results copied to the host while later runs compute) must return exactly what the
    plain path returns"""
    import workloads as wl
    from stodynprog_b200.engine import Engine
    api = _Api(product, "cuda", layout, compress=compress)
    for prob in (wl.storage_ar1(api, n_E=40, n_P=37, steps=(0.05, 0.1), item_chunk=48),
                 _searev_small(api)):
        sv = prob.solver
        sv.column_hoist = "off"       # (layout CF streams its results band by band: own test)
        J0 = np.random.default_rng(7).standard_normal(sv._state_grid_shape)
        saved = (Engine.OVERLAP_MIN_BACKUPS, Engine.OVERLAP_MIN_ITEMS)
        try:
            Engine.OVERLAP_MIN_BACKUPS, Engine.OVERLAP_MIN_ITEMS = 1 << 62, 1 << 62
            J_a, pol_a = sv.value_iteration(J0, report_time=False)
            assert not sv.engine.can_overlap_results(sv.last_tables)
            Engine.OVERLAP_MIN_BACKUPS, Engine.OVERLAP_MIN_ITEMS = 0, 0
            assert sv.engine.can_overlap_results(sv.last_tables)
            assert len(sv.engine._chunk_plan(sv.last_tables)) >= 2
            for _ in range(2):
                J_b, pol_b = sv.value_iteration(J0, report_time=False)
                assert np.array_equal(J_a, J_b) and np.array_equal(pol_a, pol_b)
            # feeding the page-locked result back in takes the no-staging upload path
            J_c, pol_c = sv.value_iteration(J_b, report_time=False)
            Engine.OVERLAP_MIN_BACKUPS, Engine.OVERLAP_MIN_ITEMS = 1 << 62, 1 << 62
            J_d, pol_d = sv.value_iteration(np.array(J_b), report_time=False)
            assert np.array_equal(J_c, J_d) and np.array_equal(pol_c, pol_d)
            # page-locked result budget exhausted: results land in pageable memory, same values
            import torch
            assert torch.from_numpy(J_d).is_pinned()
            budget = Engine.PINNED_RESULT_BUDGET
            try:
                Engine.PINNED_RESULT_BUDGET = 0
                for lim in (0, 1 << 62):
                    Engine.OVERLAP_MIN_BACKUPS, Engine.OVERLAP_MIN_ITEMS = lim, lim
                    J_e, pol_e = sv.value_iteration(np.array(J_b), report_time=False)
                    assert not torch.from_numpy(J_e).is_pinned()
                    assert np.array_equal(J_e, J_d) and np.array_equal(pol_e, pol_d)
            finally:
                Engine.PINNED_RESULT_BUDGET = budget
        finally:
            Engine.OVERLAP_MIN_BACKUPS, Engine.OVERLAP_MIN_ITEMS = saved


@gpu
@pytest.mark.parametrize("case", ["plain", "W4", "pairs", "uneven", "small_off"])
def test_column_pieces_overlapped_result_copy(product, case, monkeypatch):
    """layout CF (one band), large-sweep path of value_iteration: the column tables are tabulated
    once, every piece of columns is swept by its own launch on alternating streams, combined and
    mapped to control values by one launch (the 128-thread combine that fits next to a streaming
    CTA, or the 1024-thread one) and copied to its columns of the host arrays (2-D copies) while
    the next pieces compute - same J and policies as the plain path and as layout BF"""
    import workloads as wl
    from stodynprog_b200 import _cabi
    from stodynprog_b200.engine import Engine
    monkeypatch.setattr(Engine, "COLUMN_PIECES", (0.2, 0.5, 0.3) if case == "uneven" else (0.5, 0.25, 0.15, 0.1))
    lib = _cabi.load_library()
    lib.sdp_set_option(b"small_combine", 0 if case == "small_off" else 1)
    try:
        res = {}
        for colmode in ("off", "on"):
            api = _Api(product, "cuda", "state_minor", "auto", "on")
            sv = wl.storage_ar1(api, n_E=400, n_P=37, n_w=4 if case == "W4" else 9, steps=(0.5, 0.1)).solver
            sv.column_hoist = colmode
            sv.column_pairs = "on" if case == "pairs" else "off"
            J0 = np.random.default_rng(9).standard_normal(sv._state_grid_shape)
            monkeypatch.setattr(Engine, "OVERLAP_MIN_BACKUPS", 1 << 62)
            monkeypatch.setattr(Engine, "OVERLAP_MIN_ITEMS", 1 << 62)
            J_a, pol_a = sv.value_iteration(J0, report_time=False)
            T = sv.last_tables
            assert not sv.engine.can_overlap_results(T) and T.column == (colmode == "on")
            monkeypatch.setattr(Engine, "OVERLAP_MIN_BACKUPS", 0)
            monkeypatch.setattr(Engine, "OVERLAP_MIN_ITEMS", 0)
            assert sv.engine.can_overlap_results(T)
            if T.column:
                plan = sv.engine._chunk_plan(T)
                assert len(T.bands["tiles"]) == 1 and len(plan) == len(Engine.COLUMN_PIECES)
                assert all(ch["kind"] == "cols" for ch in plan) and T.pairs == (case == "pairs")
            for _ in range(3):
                J_b, pol_b = sv.value_iteration(J0, report_time=False)
                assert np.array_equal(J_a, J_b) and np.array_equal(pol_a, pol_b)
            J_c, pol_c = sv.value_iteration(J_b, report_time=False)       # page-locked input, second sweep
            res[colmode] = (J_a, pol_a, J_c, pol_c)
            if T.column and case == "plain":
                # page-locked result budget exhausted: the 2-D copies land in pageable memory, same values
                import torch
                budget = Engine.PINNED_RESULT_BUDGET
                try:
                    Engine.PINNED_RESULT_BUDGET = 0
                    J_e, pol_e = sv.value_iteration(np.array(J_b), report_time=False)
                    assert not torch.from_numpy(J_e).is_pinned()
                    assert np.array_equal(J_e, J_c) and np.array_equal(pol_e, pol_c)
                finally:
                    Engine.PINNED_RESULT_BUDGET = budget
        for a, b in zip(res["off"], res["on"]):
            assert np.array_equal(a.view(np.int64), b.view(np.int64))
    finally:
        lib.sdp_set_option(b"small_combine", 1)


@gpu
@pytest.mark.parametrize("bands", ["3", "5"])
def test_column_hoist_overlapped_result_copy(product, bands, monkeypatch):
    """layout CF, large-sweep path of value_iteration: the column tables are tabulated
    once, every band is swept by its own launch (its own CTA segments over the band's
    items) on alternating streams, combined and copied to the host while the next bands
    compute - same J and policies as the plain path and as layout BF"""
    import workloads as wl
    from stodynprog_b200.engine import Engine
    monkeypatch.setattr(Engine, "COLUMN_BANDS", bands)
    res = {}
    for colmode in ("off", "on"):
        api = _Api(product, "cuda", "state_minor", "auto", "on")
        sv = wl.storage_ar1(api, n_E=400, n_P=7, n_w=9, steps=(0.5, 0.1)).solver
        sv.column_hoist = colmode
        J0 = np.random.default_rng(9).standard_normal(sv._state_grid_shape)
        monkeypatch.setattr(Engine, "OVERLAP_MIN_BACKUPS", 1 << 62)
        monkeypatch.setattr(Engine, "OVERLAP_MIN_ITEMS", 1 << 62)
        J_a, pol_a = sv.value_iteration(J0, report_time=False)
        T = sv.last_tables
        assert not sv.engine.can_overlap_results(T) and T.column == (colmode == "on")
        monkeypatch.setattr(Engine, "OVERLAP_MIN_BACKUPS", 0)
        monkeypatch.setattr(Engine, "OVERLAP_MIN_ITEMS", 0)
        assert sv.engine.can_overlap_results(T)
        if T.column:
            assert len(T.bands["tiles"]) == int(bands) == len(sv.engine._chunk_plan(T))
        for _ in range(3):
            J_b, pol_b = sv.value_iteration(J0, report_time=False)
            assert np.array_equal(J_a, J_b) and np.array_equal(pol_a, pol_b)
        J_c, pol_c = sv.value_iteration(J_b, report_time=False)       # page-locked input, second sweep
        res[colmode] = (J_a, pol_a, J_c, pol_c)
    for a, b in zip(res["off"], res["on"]):
        assert np.array_equal(a.view(np.int64), b.view(np.int64))
