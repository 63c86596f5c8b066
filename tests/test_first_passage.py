"""First-passage analysis of a policy's chain: DPSolver.first_passage (sdp_first_passage of
include/sdp_b200.h).

For a target set, the recursion gives from every state the probability of reaching it within n
steps (P), the expected number of steps before reaching it (S) and the expected stage cost before
reaching it (C).  It is checked:
- against the exact chain: the scipy matrices of tests/test_forward.py (`oracle_chain`, weights as
  they are) and tests/test_sample_paths.py (`clamped_chain`), with the target rows killed, iterated
  backwards; every step of the history, both clamp settings, all three outputs;
- against identities: eval_policy for an empty target, (1, 0, 0) for the whole grid, P in [0, 1]
  and non-increasing in k with clamped weights, a converged `tol` run equal to the fixed run;
- on the GPU, bit for bit against the numpy model below (the same operations in the same order) on
  the device's own tables, run to run, across launch shapes and split calls; and statistically
  against sample_paths on config #5.

CPU suite ("model"): the host code drives the numpy model (FirstPassageFakeLib).  GPU suite
("cuda"): the real library.
"""
import ctypes

import numpy as np
import pytest

from conftest import golden
from fake_lib import _arr, _grid
from test_forward import RTOL, _case, oracle_chain, rel_l1
from test_sample_paths import ChainFakeLib, _binom_ok, _z, clamped_chain

gpu = pytest.mark.gpu


# ---------------------------------------------------------------------------
# numpy model of sdp_first_passage
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
        aP, aS, aC = np.zeros(n), np.zeros(n), np.zeros(n)
        with np.errstate(all="ignore"):
            for w in range(W):
                lam = L[:, w]

                def rec(base, k):
                    if k == d:
                        return old[base, :3]
                    a = rec(base, k + 1)
                    b = rec(base + strides[k], k + 1)
                    m = (1.0 - lam[k])[:, None]
                    return m * a + lam[k][:, None] * b

                v = rec(C[w], 0)
                aP = aP + v[:, 0] * p[w]
                aS = aS + v[:, 1] * p[w]
                aC = aC + (G[w if g_per_w else 0] + v[:, 2]) * p[w]
            new = np.zeros((n, 4))
            new[:, 0] = np.where(tmask, 1.0, aP)
            new[:, 1] = np.where(tmask, 0.0, 1.0 + aS)
            new[:, 2] = np.where(tmask, 0.0, aC)
            resid = float(np.max(np.abs(new[:, :3] - old[:, :3])))
        V = new
        if hist is not None:
            hist[step + 1] = V
    return V, resid


def outside_count(L, tmask):
    """(x, w) entries of non-target states with a weight outside [0, 1] or NaN"""
    out = ~((L >= 0.0) & (L <= 1.0))
    return int(out.any(axis=0)[:, ~tmask].sum())


def _mask_bits(words, n):
    return np.unpackbits(np.asarray(words).view(np.uint8), bitorder="little")[:n].astype(bool)


class FirstPassageFakeLib(ChainFakeLib):
    """the sdp_forward_* / sdp_chain_* models plus the model of sdp_first_passage"""

    def sdp_first_passage(self, gref, W, g_per_w, p, cell, lam, lam_plane, g, n_states, target, clamp, V_a, V_b,
                          n_steps, hist, resid_out, counters, stream):
        d, _, _, orders = _grid(gref)
        n = int(np.prod(orders))
        assert n_states == n
        strides = [int(np.prod(orders[k + 1:])) for k in range(d)]
        C = _arr(cell, W * n, ctypes.c_int32).astype(np.int64).reshape(W, n)
        L = np.stack([_arr(lam.value + 8 * k * lam_plane, W * n, ctypes.c_double).reshape(W, n)
                      for k in range(d)])
        G = _arr(g, (W if g_per_w else 1) * n, ctypes.c_double).reshape(-1, n)
        tmask = _mask_bits(_arr(target, (n + 31) // 32, ctypes.c_uint32), n)
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
            kw["_test_lib"] = FirstPassageFakeLib()
        return self.pkg.DPSolver(sys, **kw)


@pytest.fixture(scope="module", params=[pytest.param("model", id="model"),
                                        pytest.param("cuda", marks=gpu, id="cuda")])
def api(request, product):
    return _Api(product, request.param)


@pytest.fixture(scope="module")
def cuda_api(product):
    return _Api(product, "cuda")


# ---------------------------------------------------------------------------
# the cases: (solver, pol, n_steps, time_dependent, target)
# ---------------------------------------------------------------------------
def _fp_case(api, which):
    from test_wide_perturbations import _policy
    from test_parity import _toy, _two_perturbations
    if which == "storage_ar1":                             # 41 x 61, W = 9
        import workloads as wl
        solver, pol, n, td = wl.storage_ar1(api).solver, golden("storage_ar1.npz")["pi_pol"], 30, False
    elif which == "product-3x2":                           # two perturbations, W = 6
        solver = _two_perturbations(api, "mixed")
        pol, n, td = _policy(solver), 12, False
    elif which == "toy4":                                  # d = 4, W = 5
        solver = _toy(api, 4, "w", n_w=5)
        pol, n, td = _policy(solver), 12, False
    else:
        solver, pol, n, td = _case(api, which)
        n = {"inventory": 20, "searev_small": 20, "pv_storage": 240}[which]
    dims = solver._state_grid_shape
    target = np.zeros(dims, dtype=bool)
    if which == "product-3x2":
        target.reshape(-1)[::7] = True
    else:
        target[{"inventory": slice(8, None), "storage_ar1": slice(0, 6), "searev_small": slice(0, 4),
                "pv_storage": 12, "toy4": slice(0, 2)}[which]] = True
    return solver, pol, n, td, target


CASES = ["inventory", "storage_ar1", "searev_small", "pv_storage", "product-3x2", "toy4"]


def oracle_first_passage(solver, pol, target, n_steps, clamp, td):
    """[(P_k, S_k, C_k) for k = 0 .. n] of the exact chain with the target rows killed"""
    chain = clamped_chain if clamp else oracle_chain
    t = target.reshape(-1)
    P, S, C = t.astype(float), np.zeros(t.size), np.zeros(t.size)
    out = [(P, S, C)]
    fixed = None if td else chain(solver, pol)
    for k in range(n_steps - 1, -1, -1):
        A, gbar = chain(solver, pol[k], t_k=k) if td else fixed
        P, S, C = np.where(t, 1.0, A @ P), np.where(t, 0.0, 1.0 + A @ S), np.where(t, 0.0, gbar + A @ C)
        out.append((P, S, C))
    return out[::-1]


def _run(solver, pol, target, n, td, **kw):
    return solver.first_passage(pol, target, n_steps=None if td else n, report_time=False, **kw)


@pytest.mark.parametrize("clamp", [True, False], ids=["clamp", "noclamp"])
@pytest.mark.parametrize("which", CASES)
def test_against_the_exact_chain(api, which, clamp):
    solver, pol, n, td, target = _fp_case(api, which)
    dims = solver._state_grid_shape
    prob, steps, cost, info = _run(solver, pol, target, n, td, clamp=clamp, history=True)
    assert prob.shape == steps.shape == cost.shape == (n + 1,) + dims
    assert info["n_steps"] == n and not info["converged"] and info["residuals"] == []
    ref = oracle_first_passage(solver, pol, target, n, clamp, td)
    for k in range(n + 1):
        for got, want, name in zip((prob[k], steps[k], cost[k]), ref[k], "PSC"):
            assert rel_l1(got, want) <= RTOL, (which, clamp, k, name, rel_l1(got, want))
    # without history: the values of step 0, bit for bit
    p0, s0, c0, info0 = _run(solver, pol, target, n, td, clamp=clamp)
    for a, b in ((p0, prob[0]), (s0, steps[0]), (c0, cost[0])):
        assert a.shape == dims and np.array_equal(a.view(np.int64), b.view(np.int64))
    assert info0["outside_share"] == info["outside_share"] and 0.0 <= info["outside_share"] <= 1.0
    print(which, "clamp" if clamp else "noclamp", "outside share", info["outside_share"],
          "P range", float(prob[0].min()), float(prob[0].max()))


@pytest.mark.parametrize("which", ["inventory", "storage_ar1", "product-3x2"])
def test_identities(api, which):
    solver, pol, n, _, target = _fp_case(api, which)
    dims = solver._state_grid_shape
    # empty target, weights as they are: the cost is eval_policy's, bit for bit
    prob, steps, cost, _ = solver.first_passage(pol, np.zeros(dims, bool), n, clamp=False, report_time=False)
    J = solver.eval_policy(pol, n, report_time=False)
    assert np.array_equal(cost.view(np.int64), J.view(np.int64))
    assert np.all(prob == 0.0) and np.allclose(steps, n, rtol=1e-12, atol=0.0)
    # the whole grid as target: (1, 0, 0) at every step
    for clamp in (True, False):
        prob, steps, cost, info = solver.first_passage(pol, np.ones(dims, bool), n, clamp=clamp, history=True,
                                                       report_time=False)
        assert np.all(prob == 1.0) and np.all(steps == 0.0) and np.all(cost == 0.0)
        assert info["outside_share"] == 0.0
    # no step: (1_target, 0, 0)
    prob, steps, cost, info = solver.first_passage(pol, target, 0, report_time=False)
    assert np.array_equal(prob, target.astype(float)) and np.all(steps == 0) and np.all(cost == 0)
    assert info["n_steps"] == 0 and info["outside_share"] == 0.0
    # clamped weights: a probability, up to W ulp, that does not increase with k
    prob, _, _, _ = solver.first_passage(pol, target, n, history=True, report_time=False)
    W = solver.engine.build_policy_tables(solver, np.asarray(pol, dtype=float), deterministic=True).W
    eps = W * np.finfo(float).eps
    assert prob.min() >= -eps and prob.max() <= 1.0 + eps
    assert np.all(prob[:-1] >= prob[1:])


def test_tol_run_equals_the_fixed_run(api):
    """inventory, target the three lowest stock levels: every state reaches it almost surely; a
    converged tol run is the fixed run of the same length bit for bit.  The default target of the
    inventory case (levels 8 and 9) is not reached from the other levels: S grows by one per step
    and the run does not converge"""
    solver, pol, _, _, unreachable = _fp_case(api, "inventory")
    _, _, _, info = solver.first_passage(pol, unreachable, 200, tol=1e-9, check_every=25, report_time=False)
    assert not info["converged"] and info["n_steps"] == 200 and len(info["residuals"]) == 8
    assert min(info["residuals"]) >= 1.0
    target = np.zeros(solver._state_grid_shape, dtype=bool)
    target[:3] = True
    prob, steps, cost, info = solver.first_passage(pol, target, 20000, tol=1e-9, check_every=25,
                                                   report_time=False)
    m = info["n_steps"]
    assert info["converged"] and m % 25 == 0 and len(info["residuals"]) == m // 25 and m < 20000
    assert info["residuals"][-1] <= 1e-9 < info["residuals"][-2]
    p2, s2, c2, info2 = solver.first_passage(pol, target, m, report_time=False)
    for a, b in ((prob, p2), (steps, s2), (cost, c2)):
        assert np.array_equal(a.view(np.int64), b.view(np.int64))
    assert info2["outside_share"] == info["outside_share"]
    # P -> 1 everywhere; the history of a tol run stops where the run stopped
    assert np.all(np.abs(prob - 1.0) <= 1e-6), prob
    hist, _, _, info3 = solver.first_passage(pol, target, 20000, tol=1e-9, check_every=25, history=True,
                                             report_time=False)
    assert info3["n_steps"] == m and hist.shape == (m + 1,) + prob.shape
    assert np.array_equal(hist[0], prob) and np.array_equal(hist[m], target.astype(float))
    print("inventory: converged after", m, "steps; E[tau] in", float(steps.min()), float(steps.max()))


def test_argument_checks(api):
    solver, pol, n, _, target = _fp_case(api, "storage_ar1")
    dims = solver._state_grid_shape

    def run(**kw):
        args = dict(pol=pol, target=target, n_steps=3, report_time=False)
        args.update(kw)
        return solver.first_passage(**args)

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
    assert dims == target.shape
    # time-dependent system
    tsolver, tpol, _, _, ttarget = _fp_case(api, "pv_storage")
    with pytest.raises(ValueError, match=r"array `pol` should be of shape"):
        tsolver.first_passage(tpol[0], ttarget, report_time=False)
    with pytest.raises(ValueError, match="exceeds"):
        tsolver.first_passage(tpol[:10], ttarget, n_steps=11, report_time=False)
    with pytest.raises(ValueError, match="tol needs a stationary system"):
        tsolver.first_passage(tpol, ttarget, tol=1e-9, report_time=False)


# ---------------------------------------------------------------------------
# GPU: bit identity with the model, determinism, config #5 against sample_paths
# ---------------------------------------------------------------------------
def _model_on_device_tables(solver, pol, target, n, td, clamp):
    """the model, instant by instant on the device's own tables (read back): the history in the
    order of first_passage (entry k = V_k) and the outside share"""
    eng = solver.engine
    dims = solver._state_grid_shape
    N = int(np.prod(dims))
    tmask = target.reshape(-1)
    V = np.zeros((N, 4))
    V[:, 0] = tmask
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
@pytest.mark.parametrize("clamp", [True, False], ids=["clamp", "noclamp"])
@pytest.mark.parametrize("which", CASES)
def test_kernel_bit_identical_to_the_model(cuda_api, which, clamp):
    from stodynprog_b200 import _cabi
    solver, pol, n, td, target = _fp_case(cuda_api, which)
    prob, steps, cost, info = _run(solver, pol, target, n, td, clamp=clamp, history=True)
    assert _cabi.last_kernel().startswith("k_first_passage<D=%d,%s>" % (len(target.shape),
                                                                         "clamp" if clamp else "noclamp"))
    H, share = _model_on_device_tables(solver, pol, target, n, td, clamp)
    for j, got in enumerate((prob, steps, cost)):
        want = H[..., j].reshape(got.shape)
        assert np.array_equal(got.view(np.int64), want.view(np.int64)), (which, clamp, "PSC"[j])
    assert info["outside_share"] == share
    print(which, "clamp" if clamp else "noclamp", "outside share", share)


@gpu
def test_runs_launch_shapes_and_split_calls(cuda_api):
    import torch
    from stodynprog_b200 import _cabi
    solver, pol, _, _, target = _fp_case(cuda_api, "storage_ar1")
    eng = solver.engine
    lib = eng.lib
    P = eng.build_policy_tables(solver, np.asarray(pol, dtype=float), deterministic=True)
    N = P.n_states
    mask = eng.to_device(solver._target_mask(target))
    V0 = np.zeros((N, 4))
    V0[:, 0] = target.reshape(-1)
    n = 41

    def run(threads, split, clamp=True):
        lib.sdp_set_option(b"fp_threads", threads)
        a = eng.to_device(V0.reshape(-1))
        b = torch.empty_like(a)
        cnt = torch.zeros(1, dtype=torch.int64, device=eng.device)
        res = torch.zeros(1, dtype=torch.float64, device=eng.device)
        hist = torch.empty((n + 1) * N * 4, dtype=torch.float64, device=eng.device)
        done = 0
        for k in split:
            out = eng.first_passage(P, mask, clamp, a, b, k, hist=hist[done * N * 4:(done + k + 1) * N * 4],
                                    resid_out=res, counters=cnt)
            if out is b:
                a, b = b, a
            done += k
        name = _cabi.last_kernel()
        return [t.cpu().numpy() for t in (a.view(torch.int64), hist.view(torch.int64), res.view(torch.int64))], \
            int(cnt.cpu().numpy()[0]) // len(split), name

    try:
        ref, cnt, name = run(0, [n])
        assert name == "k_first_passage<D=2,clamp>, 256 threads", name
        res = ref[2].view(np.float64)[0]
        assert res > 0.0 and ref[0].view(np.float64).reshape(N, 4)[:, 3].max() == 0.0
        for threads, split in [(0, [n]), (96, [n]), (1024, [n]), (0, [17, 24]), (160, [1, 20, 20])]:
            got, c, name = run(threads, split)
            assert str(threads or 256) in name
            assert c == cnt, (threads, split)
            for a, b in zip(ref, got):
                assert np.array_equal(a, b), (threads, split)
    finally:
        lib.sdp_set_option(b"fp_threads", 0)


@gpu
def test_nan_makes_the_residual_nan(cuda_api):
    """a NaN value at a corner reaches the residual: a tol run never reports convergence on it"""
    import torch
    solver, pol, _, _, target = _fp_case(cuda_api, "inventory")
    eng = solver.engine
    P = eng.build_policy_tables(solver, np.asarray(pol, dtype=float), deterministic=True)
    N = P.n_states
    V0 = np.zeros((N, 4))
    V0[:, 0] = target.reshape(-1)
    V0[N // 2, 1] = np.nan
    a = eng.to_device(V0.reshape(-1))
    b = torch.empty_like(a)
    res = torch.zeros(1, dtype=torch.float64, device=eng.device)
    eng.first_passage(P, eng.to_device(solver._target_mask(target)), True, a, b, 3, resid_out=res)
    assert np.isnan(res.cpu().numpy()[0])


@gpu
def test_config5_against_sample_paths(cuda_api):
    """config #5 (2000 x 500, W = 9), target the empty storage (axis-0 index 0): the hit frequency
    of 1e5 sampled paths against P (binomial tails) and their mean of min(tau, n) against S (5
    standard errors, Bonferroni over the four checks), from one multi-index and from a start
    distribution.  The start is the full storage on the middle column, the horizon the first n at
    which P from there reaches 1/2 (read from a history of 100 steps)"""
    import workloads as wl
    prob_ = wl.storage_ar1_large(cuda_api)
    solver = prob_.solver
    _, pol = solver.value_iteration(prob_.J0, report_time=False)
    dims = solver._state_grid_shape
    target = np.zeros(dims, dtype=bool)
    target[0] = True
    start = (dims[0] - 1, dims[1] // 2)
    N, M, K = 100, 100000, 4
    hist, _, _, _ = solver.first_passage(pol, target, N, history=True, report_time=False)
    law = hist[::-1][(slice(None),) + start]           # P(tau <= j) from the start, j = 0 .. N
    assert np.all(np.diff(law) >= 0.0) and law[-1] >= 0.5, law
    n = int(np.argmax(law >= 0.5))
    prob, steps, _, info = solver.first_passage(pol, target, n, report_time=False)
    assert np.array_equal(prob, hist[N - n])           # a history entry is the shorter run, bit for bit
    p_s, s_s = float(prob[start]), float(steps[start])
    print("config #5: start", start, "horizon", n, "P", p_s, "S", s_s, "outside share", info["outside_share"])
    assert 0.05 < p_s < 0.95
    # the start distribution: random weights on the states whose P lies in [0.1, 0.9]
    mu0 = np.random.default_rng(8).random(dims) * ((prob >= 0.1) & (prob <= 0.9))
    p_mu = float((mu0 * prob).sum() / mu0.sum())
    s_mu = float((mu0 * steps).sum() / mu0.sum())
    print("config #5: start distribution over", int((mu0 > 0).sum()), "states, P", p_mu, "S", s_mu)
    assert 0.05 < p_mu < 0.95
    for start_, p_x, s_x, seed in ((start, p_s, s_s, 31), (mu0, p_mu, s_mu, 32)):
        _, sp_info = solver.sample_paths(pol, start_, n, M, seed=seed, target=target, report_time=False)
        h = sp_info["hit_step"]
        hits = int((h >= 0).sum())
        assert _binom_ok(hits, M, p_x, K), (hits / M, p_x)
        tau_n = np.where(h < 0, n, h).astype(float)
        se = tau_n.std() / np.sqrt(M)
        assert abs(tau_n.mean() - s_x) <= _z(K) * se, (tau_n.mean(), s_x, se)
        print("sampled: hit", hits / M, "mean min(tau, n)", tau_n.mean(), "se", se)
