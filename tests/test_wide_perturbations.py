"""Wide perturbation grids, d = 4 in the policy-analysis paths, and the tail paths of the kernels.

The other suites use perturbation grids of at most 9 nodes.  The sweeps accept up to 4096, layout
AF up to 128, and the analysis paths (propagate_distribution, stationary_distribution,
sample_paths) set no limit of their own.  The cases here sit on the thresholds where the
kernels change: the register slots of layouts BF/CF (W <= 9), the row budget of the AF hoist
(capped at 32 rows up to W = 20 for d = 2; fewer than 2 rows, so the plain AF kernel, from W = 126
for d = 3), the shared-memory cap of layout AF (W <= 128), the tail loops of the state-minor
kernels (W or u_count * W not a multiple of the block), the 200 KB fit of the TMA rings, the long
rows of the forward operator (more than SDP_FWD_PIECE entries) and the node search of the path
sampler.

Like the other suites, the tests run with backend "model" (tests/fake_lib.py and its extensions,
CPU suite) and "cuda" (marked gpu).  The references are the oracle port for the sweeps, the scipy
chain of tests/test_forward.py for the forward operator, and the numpy twin tests/chain_twin.py
for the sampler.
"""
import ctypes

import numpy as np
import pytest
import scipy.stats as stats

import chain_twin
from conftest import rel_err
from test_forward import RTOL, oracle_propagate, rel_l1
from test_parity import J_RTOL, _Api, _same_bits, _separable, _toy, _two_perturbations
from test_sample_paths import _Api as _ChainApi, _binom_ok, _twin_run, _z, exact_moments
from stodynprog_b200 import _cabi

gpu = pytest.mark.gpu
BACKENDS = [pytest.param("model", id="model"), pytest.param("cuda", marks=gpu, id="cuda")]

# (table_layout, tabulate, table_compress, column_hoist) of the layouts asked for
LAYOUTS = {"A": ("control_minor", "auto", "off", "off"), "B": ("state_minor", "auto", "off", "off"),
           "AF": ("control_minor", "auto", "auto", "off"), "auto": ("state_minor", "auto", "auto", "auto")}
# the factored split (u_mask) of the _separable systems
MASKS = {"uw": 1, "uww": 1, "wuw": 2, "wwu": 4}


def _system(api, which, W):
    """toy<d>: the _toy system (w-dependent cost, dense tables; W = 0: deterministic);
    otherwise _separable(which) with an (x,u) + (x,w) split"""
    if which.startswith("toy"):
        return _toy(api, int(which[3:]), "w", n_w=W)
    return _separable(api, tuple(which), n_w=W)


# ---------------------------------------------------------------------------
# 1. sweep parity at wide W against the oracle port
# ---------------------------------------------------------------------------
def _sweep_cases():
    cases = []

    def add(which, W, layouts):
        for lay in layouts:
            cases.append((which, W, lay))

    for d in (1, 2, 4):                                   # W = 1, deterministic (expect = 0)
        add("toy%d" % d, 0, ["A", "B"] + (["auto"] if d < 4 else []))
    add("toy2", 1, ["A", "B", "AF", "auto"])              # W = 1, one node of probability 1
    add("uw", 1, ["AF", "auto"])
    for W in (2, 10, 17, 20, 21, 33, 64, 125, 126, 128, 129, 257):
        add("uw", W, ["AF", "auto"])
        add("uww", W, ["AF"])
        add("toy2", W, ["A", "B"])
    for W in (10, 33, 128):
        add("wuw", W, ["AF"])
    for W in (10, 33):
        add("toy4", W, ["A", "B"])
    for W in (1000, 4096):                                # large W on small grids, d <= 2
        add("toy1", W, ["A", "B"])
        add("uw", W, ["AF", "auto"])
    return cases


SWEEP_CASES = _sweep_cases()
_PORT = {}


def _j0(sv):
    J0 = np.random.default_rng(17).standard_normal(sv._state_grid_shape)
    J0.reshape(-1)[0] = np.nan         # NaN where a next state's corner reaches the first node
    return J0


def _port_results(port, which, W):
    """value iteration, policy evaluation (plain and relative) and 3 steps of policy iteration
    of the oracle port, computed once per system"""
    key = (which, W)
    if key not in _PORT:
        so = _system(port, which, W)
        with np.errstate(invalid="ignore"):
            Jo, polo = so.value_iteration(_j0(so))
        out = {"vi": (Jo, polo)}
        if W:
            out["eval"] = so.eval_policy(polo, 7)
            out["rel"] = so.eval_policy(polo, 7, rel_dp=True)
            out["pi"] = so.policy_iteration(polo, 4, 3, rel_dp=True)
        _PORT[key] = out
    return _PORT[key]


def _expected_layout(which, W, lay):
    d = 1 if which == "toy1" else (2 if which in ("toy2", "uw") else (4 if which == "toy4" else 3))
    factorable = not which.startswith("toy") and 1 < W and d in (2, 3)
    if lay == "A" or (lay == "AF" and not (factorable and W <= _cabi.FACTORED_MAX_W_SMEM)):
        return "control_minor", d
    if lay == "AF":
        return "control_minor_factored", d
    if lay == "B" or not (factorable and W <= _cabi.FACTORED_MAX_W_REG):
        return "state_minor", d
    return "state_minor_factored", d       # (7 rows of axis 0: too few for layout CF)


def _expected_kernel(which, W, lay, layout, d):
    if layout == "control_minor":
        return "k_sweep<%d," % d
    if layout == "state_minor":
        return "k_sweep_tiled"
    if layout == "state_minor_factored":
        return "k_sweep_fact_tiled<%d,%d," % (d, MASKS[which])
    if MASKS[which] != 1:
        return "k_sweep_fact<%d,%d," % (d, MASKS[which])
    if W <= _cabi.FACTORED_MAX_W_REG:
        return "k_sweep_fact_hoist_c<%d," % d
    if d == 3 and W >= 126:            # fewer than 2 rows of the hoisted table fit 44 KB
        return "k_sweep_fact<3,1,"
    return "k_sweep_fact_hoist<%d," % d


def _close(J, Jo):
    nan = np.isnan(J)
    return np.array_equal(nan, np.isnan(Jo)) and rel_err(np.where(nan, 0, J), np.where(nan, 0, Jo)) <= J_RTOL


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("which,W,lay", SWEEP_CASES,
                         ids=["%s-W%d-%s" % c if c[1] else "%s-det-%s" % (c[0], c[2]) for c in SWEEP_CASES])
def test_sweeps_against_port(product, port, backend, which, W, lay):
    """value iteration (NaN in J included), policy evaluation with and without relative DP and
    policy iteration against the oracle port; the plan the sweep used"""
    sv = _system(_Api(product, backend, *LAYOUTS[lay]), which, W)
    ref = _port_results(port, which, W)
    J, pol = sv.value_iteration(_j0(sv), report_time=False)
    name = _cabi.last_kernel() if backend == "cuda" else None
    T = sv.last_tables
    layout, d = _expected_layout(which, W, lay)
    assert T.W == max(W, 1) and T.expect == (1 if W else 0)
    assert T.layout_name == layout, (T.layout_name, layout)
    if name is not None:
        assert name.startswith(_expected_kernel(which, W, lay, layout, d)), name
    Jo, polo = ref["vi"]
    assert np.array_equal(pol, polo)
    assert _close(J, Jo)
    if not W:
        return
    Je = sv.eval_policy(pol, 7, report_time=False)
    assert rel_err(Je, ref["eval"]) <= J_RTOL
    Jr, jr = sv.eval_policy(pol, 7, rel_dp=True, report_time=False)
    Jro, jro = ref["rel"]
    assert abs(jr - jro) <= J_RTOL * abs(jro)
    assert np.max(np.abs(Jr - Jro)) <= J_RTOL * max(np.max(np.abs(Jro)), 1e-300)
    (Jp, jp), polp = sv.policy_iteration(pol, 4, 3, rel_dp=True)
    (Jpo, jpo), polpo = ref["pi"]
    assert np.array_equal(polp, polpo) and abs(jp - jpo) <= J_RTOL * abs(jpo)
    assert np.max(np.abs(Jp - Jpo)) <= J_RTOL * max(np.max(np.abs(Jpo)), 1e-300)


def test_wide_W_limits(product):
    """the sweeps refuse more than 4096 nodes; table_compress='on' refuses layout AF beyond 128"""
    with pytest.raises(ValueError, match="4096"):
        _system(_Api(product, "model", *LAYOUTS["A"]), "toy1", 4097).value_iteration(
            np.zeros(6), report_time=False)
    sv = _system(_Api(product, "model", "control_minor", "auto", "on", "off"), "uw", 129)
    with pytest.raises(ValueError, match="table_compress='on'"):
        sv.value_iteration(np.zeros(sv._state_grid_shape), report_time=False)


# ---------------------------------------------------------------------------
# 2. kernel variants at wide W: bit-identical to each other
# ---------------------------------------------------------------------------
def _tiny4(api, W, **kw):
    """d = 4 on 3x2x2x2 = 24 states, 5 controls per state, cost depending on w (g_per_w)"""
    def dyn(x0, x1, x2, x3, u, w):
        return (0.8 * x0 + 0.5 * u + 0.3 * w, 0.7 * x1 + 0.2 * u - 0.2 * w, 0.9 * x2 + 0.4 * w,
                0.6 * x3 + 0.3 * u * w)

    def box(x0, x1, x2, x3):
        return ((-1.0, 1.0),)

    def cost(x0, x1, x2, x3, u, w):
        return x0 ** 2 + x1 ** 2 + 0.5 * x2 ** 2 + 0.3 * x3 ** 2 + 0.1 * u ** 2 + 0.05 * w * u

    sys = api.SysDescription((4, 1, 1), name='tiny4')
    sys.dyn, sys.control_box, sys.cost = dyn, box, cost
    sys.perturb_laws = [stats.norm(0, 0.4)]
    sv = api.DPSolver(sys, **kw)
    sv.discretize_state(-1.0, 1.0, 3, -1.0, 1.0, 2, -1.0, 1.0, 2, -1.0, 1.0, 2)
    sv.discretize_perturb(-1.0, 1.0, W)
    sv.control_steps = (0.5,)
    return sv


DEFAULTS = dict(tma=1, tma_rows=8, tma_stages=2, tma_warps=4, rb=4, wb=1, upl=4, hoist=1, hoist_const=1,
                hoist_upl=2)
B_SETTINGS = [dict(tma=0, wb=1), dict(tma=0, wb=2), dict(tma=0, wb=3), dict(tma=0, wb=5),
              dict(tma=2, rb=2), dict(tma=2, rb=4), dict(tma=2, rb=8),
              dict(tma=1, tma_rows=8, tma_stages=2, tma_warps=4), dict(tma=1, tma_rows=4, tma_stages=3, tma_warps=8),
              dict(tma=1, tma_rows=8, tma_stages=5, tma_warps=2), dict(tma=1, tma_rows=8, tma_stages=16, tma_warps=8)]
AF_SETTINGS = [dict(hoist=h, hoist_const=c, hoist_upl=u, upl=u)
               for h in (1, 0) for c in (1, 0) for u in (2, 4)]


def _opt(lib, **kw):
    for k, v in kw.items():
        _cabi.check(lib.sdp_set_option(k.encode(), int(v)), "sdp_set_option")


def _variants_agree(lib, sv, settings):
    J0 = np.random.default_rng(8).standard_normal(sv._state_grid_shape)
    ref, names = None, []
    for st in settings:
        _opt(lib, **st)
        J, pol = sv.value_iteration(J0, report_time=False)
        names.append(_cabi.last_kernel())
        if ref is None:
            ref = (J, pol)
        assert _same_bits(J, ref[0]) and _same_bits(pol, ref[1]), (st, names[-1])
    return names


@gpu
@pytest.mark.parametrize("W", [7, 10, 33, 257])
def test_kernel_variants_at_wide_W(product, W):
    """layout B: LDG kernel with every W block (tail loops), pipelined kernel with every row block,
    TMA rings with partial last stages and items of fewer rows than a stage (tiny4: items of 1
    control); layout A with both lane widths; layout AF with and without the hoist, the
    constant-W kernel and both lane widths"""
    lib = _cabi.load_library()
    try:
        for sv in (_toy(_Api(product, "cuda", "state_minor", "auto", "off"), 2, "w", n_w=W, item_chunk=8),
                   _tiny4(_Api(product, "cuda", "state_minor", "auto", "off"), W, item_chunk=4)):
            names = _variants_agree(lib, sv, B_SETTINGS)
            assert sv.last_tables.layout_name == "state_minor"
            assert names[1].startswith("k_sweep_tiled<") and names[4].startswith("k_sweep_tiled_pipe<")
        for sv in (_toy(_Api(product, "cuda", "control_minor", "auto", "off"), 2, "w", n_w=W, item_chunk=8),
                   _tiny4(_Api(product, "cuda", "control_minor", "auto", "off"), W, item_chunk=4)):
            _variants_agree(lib, sv, [dict(upl=4), dict(upl=2)])
        if W <= _cabi.FACTORED_MAX_W_SMEM:
            for which in ("uw", "uww"):
                sv = _separable(_Api(product, "cuda", "control_minor", "auto", "on"), tuple(which), n_w=W)
                names = _variants_agree(lib, sv, AF_SETTINGS)
                assert sv.last_tables.layout_name == "control_minor_factored"
                assert any(n.startswith("k_sweep_fact<") for n in names)
    finally:
        _opt(lib, **DEFAULTS)


@gpu
def test_tma_ring_fit(product):
    """16 stages of 8 rows of 5 planes (d = 4, g_per_w) and 8 warps: the rings shrink to one warp
    and fit 200 KB at W = 2000; at W = 4096 the 32 KB of node probabilities leave no room and the
    LDG kernel runs.  J and argmin as the LDG kernel's"""
    lib = _cabi.load_library()
    try:
        for W, fits in ((2000, True), (4096, False)):
            sv = _tiny4(_Api(product, "cuda", "state_minor", "auto", "off"), W)
            names = _variants_agree(lib, sv, [dict(tma=0, wb=1),
                                              dict(tma=1, tma_rows=8, tma_stages=16, tma_warps=8)])
            assert sv.last_tables.g_per_w == 1
            if fits:
                assert names[1] == "k_sweep_tiled_tma<4,8> [16 stages, 32 threads]", names[1]
            else:
                assert names[1] == "k_sweep_tiled<4,1>", names[1]
    finally:
        _opt(lib, **DEFAULTS)


# ---------------------------------------------------------------------------
# 3. forward operator and path sampler: d = 4, wide W, product grids, long rows
# ---------------------------------------------------------------------------
def _two_normal_perturbations(api, n1, n2):
    """d = 2, one control, two independent normal perturbations on n1 x n2 nodes"""
    def dyn(x0, x1, u, w1, w2):
        return (0.8 * x0 + 0.4 * u + 0.3 * w1, 0.7 * x1 + 0.2 * u * w2 + 0.1 * w1)

    def box(x0, x1):
        return ((-1.0, 1.0),)

    def cost(x0, x1, u, w1, w2):
        return x0 ** 2 + 0.5 * x1 ** 2 + 0.1 * u ** 2 + 0.05 * w1 * u - 0.02 * w2

    sys = api.SysDescription((2, 1, 2), name='two normal perturbations')
    sys.dyn, sys.control_box, sys.cost = dyn, box, cost
    sys.perturb_laws = [stats.norm(0, 0.5), stats.norm(0, 0.3)]
    sv = api.DPSolver(sys)
    sv.discretize_state(-1.0, 2.0, 6, -1.0, 1.5, 5)
    sv.discretize_perturb(-0.9, 0.9, n1, -0.6, 0.6, n2)
    sv.control_steps = (2.0 / 23,)
    return sv


def _policy(sv):
    """a fixed admissible policy: an irregular pattern of controls inside [-0.9, 0.9]"""
    n = int(np.prod(sv._state_grid_shape))
    return (0.9 * np.sin(1.7 * np.arange(n))).reshape(sv._state_grid_shape + (1,))


def _analysis_case(api, which):
    if which == "toy4-det":
        return _toy(api, 4, "w", n_w=0)
    if which == "toy4-W33":
        return _toy(api, 4, "w", n_w=33)
    if which == "toy2-W4096":
        return _toy(api, 2, "w", n_w=4096)
    if which == "product-3x2":
        return _two_perturbations(api, "mixed")
    if which == "product-16x16":
        return _two_normal_perturbations(api, 16, 16)
    raise KeyError(which)


ANALYSIS_CASES = ["toy4-det", "toy4-W33", "toy2-W4096", "product-3x2", "product-16x16"]


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("which", ANALYSIS_CASES)
def test_propagate_against_scipy_oracle(product, backend, which):
    sv = _analysis_case(_ChainApi(product, backend), which)
    pol = _policy(sv)
    mu0 = np.random.default_rng(2).random(sv._state_grid_shape)
    n = 12
    mu, cost = sv.propagate_distribution(pol, mu0, n_steps=n, report_time=False)
    mu_o, cost_o = oracle_propagate(sv, pol, mu0, n)
    assert rel_l1(mu, mu_o) <= RTOL and rel_l1(cost, cost_o) <= RTOL
    hist, cost_h = sv.propagate_distribution(pol, mu0, n_steps=4, history=True, report_time=False)
    for k in range(5):
        assert rel_l1(hist[k], oracle_propagate(sv, pol, mu0, k)[0]) <= RTOL
    assert rel_l1(cost_h, cost_o[:4]) <= RTOL


def _funnel(api, n, W):
    """d = 1, n states on [0, 1]: every next state is grid node n // 2 exactly, so the rows of
    nodes n // 2 and n // 2 + 1 hold n * W entries each (weights 1 and 0)"""
    node = np.linspace(0.0, 1.0, n)[n // 2]

    def dyn(x, u, w):
        return (0.0 * (x + u + w) + node,)

    def box(x):
        return ((0.0, 1.0),)

    def cost(x, u, w):
        return x ** 2 + 0.3 * u + 0.1 * w * x

    sys = api.SysDescription((1, 1, 1), name='funnel')
    sys.dyn, sys.control_box, sys.cost = dyn, box, cost
    sys.perturb_laws = [stats.norm(0, 1.0)]
    sv = api.DPSolver(sys)
    sv.discretize_state(0.0, 1.0, n)
    sv.discretize_perturb(-2.0, 2.0, W)
    sv.control_steps = (0.5,)
    return sv


@pytest.mark.parametrize("backend", BACKENDS)
@pytest.mark.parametrize("n,W,pieces", [(32, 32, 0), (25, 41, 2), (32, 64, 2), (3, 683, 3)],
                         ids=["1024", "1025", "2048", "2049"])
def test_long_rows_of_the_forward_operator(product, backend, n, W, pieces):
    """rows of n*W = 1024 entries stay on the team path; 1025, 2048 and 2049 entries make 2, 2 and 3
    pieces per row, summed in piece order whatever the launch"""
    import torch
    sv = _funnel(_ChainApi(product, backend), n, W)
    pol = np.linspace(0.0, 1.0, n).reshape(n, 1)
    F = sv._forward_operator(pol)
    assert F.n_pieces == 2 * pieces
    mu0 = np.random.default_rng(n + W).random(n)
    mu, cost = sv.propagate_distribution(pol, mu0, n_steps=3, report_time=False)
    mu_o, cost_o = oracle_propagate(sv, pol, mu0, 3)
    assert rel_l1(mu, mu_o) <= RTOL and rel_l1(cost, cost_o) <= RTOL
    assert abs(mu[n // 2] - mu0.sum()) <= 1e-12 * mu0.sum()
    mu2, cost2 = sv.propagate_distribution(pol, mu0, n_steps=3, report_time=False)
    assert _same_bits(mu, mu2) and _same_bits(cost, cost2)
    # one launch of 3 steps against 3 launches of 1 step on the same operator
    eng = sv.engine
    a = eng.to_device(mu0)
    b = torch.empty_like(a)
    c = torch.zeros(3, dtype=torch.float64, device=eng.device)
    for k in range(3):
        out = eng.forward_steps(F, a, b, 1, c[k:k + 1])
        a, b = out, (b if out is a else a)
    assert _same_bits(a.cpu().numpy(), mu) and _same_bits(c.cpu().numpy(), cost)


def _sampled_case(api, which):
    if which == "zero-p":
        return _zero_p(api)
    if which == "W33":
        return _toy(api, 2, "w", n_w=33)
    if which == "W4096":
        return _toy(api, 1, "w", n_w=4096)
    if which == "toy4":
        return _toy(api, 4, "w", n_w=5)
    return _analysis_case(api, which)


def _zero_p(api):
    """d = 1 on 11 nodes of [0, 10], 9 perturbation nodes of which the first, the middle and the
    last have probability 0: those send the state to node 10, which nothing else reaches"""
    poison = (0, 4, 8)

    def dyn(x, u, w):
        normal = np.clip(0.5 * x + u + 0.5 * w, 0.0, 9.0)
        return (np.where(np.isin(w, [float(i) for i in poison]), 10.0, normal),)

    def box(x):
        return ((0.0, 3.0),)

    def cost(x, u, w):
        return x + 0.2 * u + 0.1 * w

    law = stats.rv_discrete(values=(np.arange(9), np.where(np.isin(np.arange(9), poison), 0.0, 1.0 / 6)))
    sys = api.SysDescription((1, 1, 1), name='zero-probability nodes')
    sys.dyn, sys.control_box, sys.cost = dyn, box, cost
    sys.perturb_laws = [law.freeze()]
    sv = api.DPSolver(sys)
    sv.discretize_state(0.0, 10.0, 11)
    sv.discretize_perturb(0, 8, 9)
    sv.control_steps = (0.5,)
    return sv


@pytest.mark.parametrize("backend", BACKENDS)
def test_zero_probability_nodes_are_never_drawn(product, backend):
    sv = _zero_p(_ChainApi(product, backend))
    assert list(np.flatnonzero(sv.perturb_proba[0] == 0)) == [0, 4, 8]
    pol = (np.arange(11) % 4 * 0.5).reshape(11, 1)
    start = np.ones(11)
    start[10] = 0.0
    target = np.zeros(11, dtype=bool)
    target[10] = True
    n_steps = 40
    _, info = sv.sample_paths(pol, start, n_steps, 5000, seed=21, target=target, record=list(range(n_steps + 1)),
                              report_time=False)
    assert info["states"].max() <= 9 and np.all(info["hit_step"] == -1)
    assert len(np.unique(info["states"])) >= 9       # the paths do move around


@gpu
@pytest.mark.parametrize("which", ["toy4", "W33", "W4096", "product-16x16", "zero-p"])
def test_kernel_bit_identical_to_the_twin(product, which):
    """as tests/test_sample_paths.py: the packed records, then total, hit step, recorded and final
    states and the counters, bit for bit; d = 4 draws its fourth coordinate from a third Philox call"""
    sv = _sampled_case(_ChainApi(product, "cuda"), which)
    pol = _policy(sv) if which != "zero-p" else (np.arange(11) % 4 * 0.5).reshape(11, 1)
    dims = sv._state_grid_shape
    start = np.random.default_rng(4).random(dims)
    target = np.zeros(dims, dtype=bool)
    target.reshape(-1)[::7] = True
    M, seed, n_steps = 4096, 987654321, 30
    steps = [0, 11, n_steps]
    total, info = sv.sample_paths(pol, start, n_steps, M, seed=seed, target=target, record=steps,
                                  report_time=False)
    assert _cabi.last_kernel().startswith("k_chain_sample<D=%d>" % len(dims))
    eng = sv.engine
    P = eng.build_policy_tables(sv, np.asarray(pol, dtype=float), deterministic=True)
    C = eng.chain_tables(P)
    d = P.grid.d
    planes = chain_twin.pack(d, P.W, P.g_per_w, P.n_states, P.cell.cpu().numpy()[:P.W * P.n_states],
                             P.lam.cpu().numpy()[:d * P.lam_plane], P.g.cpu().numpy())
    assert np.array_equal(planes.view(np.int64), C.rec.cpu().numpy().reshape(planes.shape).view(np.int64))
    st, tot, h, cnt, rec = _twin_run(eng, C, n_steps, 0, seed, True, np.zeros(M, np.int32), np.zeros(M),
                                     np.zeros(M, np.int32), start_cdf=np.cumsum(start.reshape(-1)),
                                     target=sv._target_mask(target).view(np.uint32), rec_steps=steps)
    assert np.array_equal(total.view(np.int64), tot.view(np.int64))
    assert np.array_equal(info["hit_step"], h) and np.array_equal(info["final_state"], st)
    assert np.array_equal(info["states"], rec)
    assert info["clamped_share"] == cnt[0] / (M * n_steps) and info["nan_transitions"] == cnt[1]


@pytest.mark.parametrize("backend", BACKENDS)
def test_d4_statistics_against_the_exact_chain(product, backend):
    """d = 4 (toy, W = 5): state distribution at recorded steps, mean total cost and hit probability
    within 5 standard errors (Bonferroni) of the exact clamped chain"""
    sv = _toy(_ChainApi(product, backend), 4, "w", n_w=5)
    pol = _policy(sv)
    dims = sv._state_grid_shape
    start = np.zeros(dims)
    start[dims[0] // 2:] = np.random.default_rng(1).random((dims[0] - dims[0] // 2,) + dims[1:])
    target = np.zeros(dims, dtype=bool)
    target[:2] = True
    M, n_steps = 20000, 12
    steps = [0, 1, n_steps // 2, n_steps]
    total, info = sv.sample_paths(pol, start, n_steps, M, seed=13, target=target, record=steps,
                                  report_time=False)
    mus, cost, p_hit = exact_moments(sv, pol, n_steps, False, start, target, steps)
    n = start.size
    K = len(steps) * n + 2
    for j, k in enumerate(steps):
        counts = np.bincount(info["states"][j], minlength=n)
        assert _binom_ok(counts, M, mus[j], K).all(), k
    se = total.std() / np.sqrt(M)
    assert abs(total.mean() - cost) <= _z(K) * se + 1e-9 * abs(cost), (total.mean(), cost, se)
    assert _binom_ok(int((info["hit_step"] >= 0).sum()), M, p_hit, K)
    print("d = 4: clamped share", info["clamped_share"], "hit", np.mean(info["hit_step"] >= 0), p_hit)


# ---------------------------------------------------------------------------
# 4. the sampler's shared-memory bound: node CDF (dynamic) + the kernel's static shared memory
#    within the 48 KB of a launch without an opt-in
# ---------------------------------------------------------------------------
@gpu
def test_sampler_node_limit(product):
    """through the C ABI on a 2-state grid: W = 6144 (48 KB of CDF alone) is refused with
    SDP_EINVAL before any launch, and the message gives the bound; the bound itself launches and
    matches the twin, one node more is refused"""
    import re
    import torch
    from stodynprog_b200.engine import Engine
    eng = Engine()
    grid = _cabi.make_grid([np.array([0.0, 1.0])])
    n, M, n_steps, seed = 2, 2048, 5, 77

    def run(W):
        rng = np.random.default_rng(W)
        p = rng.random(W)
        p[::5] = 0.0
        cdf = np.cumsum(p / p.sum())
        rec_h = chain_twin.pack(1, W, 1, n, np.zeros(n * W, np.int32), rng.random(n * W), rng.standard_normal(n * W))
        cdf_d, rec = eng.to_device(cdf), eng.to_device(np.ascontiguousarray(rec_h.reshape(-1)))
        state = eng.to_device(np.arange(M, dtype=np.int32) % n)
        total = torch.zeros(M, dtype=torch.float64, device=eng.device)
        hit = torch.zeros(M, dtype=torch.int32, device=eng.device)
        cnt = torch.zeros(2, dtype=torch.int64, device=eng.device)
        launches = _cabi.launch_count()
        rc = eng.lib.sdp_chain_sample(ctypes.byref(grid), W, eng._ptr(cdf_d), eng._ptr(rec), M, n_steps, 0, seed, 1,
                                      None, None, None, 0, eng._ptr(state), eng._ptr(total), eng._ptr(hit), None,
                                      eng._ptr(cnt), eng.stream)
        if rc:
            assert rc == -1 and _cabi.launch_count() == launches       # SDP_EINVAL, nothing launched
            return eng.lib.sdp_last_error().decode()
        st, tot, h, c = np.arange(M, dtype=np.int32) % n, np.zeros(M), np.zeros(M, np.int32), [0, 0]
        chain_twin.sample([1], W, cdf, rec_h, n, n_steps, 0, seed, True, st, tot, h, c)
        assert np.array_equal(state.cpu().numpy(), st)
        assert np.array_equal(total.cpu().numpy().view(np.int64), tot.view(np.int64))
        assert np.array_equal(cnt.cpu().numpy(), c)
        return None

    msg = run(6144)
    m = re.search(r"W > (\d+) nodes", msg or "")
    assert m, msg
    w_max = int(m.group(1))
    print("sampler node bound", w_max, msg)
    assert 5000 < w_max < 6144
    assert run(w_max) is None
    assert run(w_max + 1) == msg
