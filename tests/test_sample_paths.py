"""Sample paths of a policy's chain: DPSolver.sample_paths (sdp_chain_pack / sdp_chain_sample of
include/sdp_b200.h).

The sampler is checked two ways:
- exactly, against the numpy twin of tests/chain_twin.py (same Philox bits, same fp64 operations):
  the CPU suite ("model") drives the host code through the twin, the GPU suite compares the
  kernels with it bit for bit;
- statistically, against the exact chain: the scipy matrix of tests/test_forward.py with the
  interpolation weights clamped to [0, 1], as the sampler clamps them.  The distribution of the
  state at the recorded steps, the mean total cost and the probability of reaching a target set
  must agree within 5 standard errors with a Bonferroni factor (binomial tails for frequencies).
  The seeds are fixed, so these tests are deterministic.
"""
import ctypes

import numpy as np
import pytest
import scipy.sparse as sp
from scipy import stats

import chain_twin
from conftest import golden
from fake_lib import _arr, _grid
from oracle import oracle as oc
from stodynprog_b200 import _cabi
from test_forward import ForwardFakeLib, _case, oracle_chain

gpu = pytest.mark.gpu


class ChainFakeLib(ForwardFakeLib):
    """the sdp_forward_* model plus the twin of sdp_chain_pack / sdp_chain_sample"""

    def sdp_chain_pack(self, gref, W, g_per_w, cell, lam, lam_plane, g, n, rec, stream):
        d = _grid(gref)[0]
        C = _arr(cell, W * n, ctypes.c_int32)
        L = np.stack([_arr(lam.value + 8 * k * lam_plane, W * n, ctypes.c_double) for k in range(d)])
        G = _arr(g, (W if g_per_w else 1) * n, ctypes.c_double)
        R = _cabi.chain_rec(d)
        _arr(rec, n * W * R, ctypes.c_double)[:] = chain_twin.pack(d, W, g_per_w, n, C, L, G).reshape(-1)
        self.launches += 1
        return 0

    def sdp_chain_sample(self, gref, W, cdf, rec, M, n_steps, step0, seed, fresh, start_cdf, target, rec_steps,
                         n_rec, state, total, hit, rec_out, counters, stream):
        d, _, _, orders = _grid(gref)
        n = int(np.prod(orders))
        strides = [int(np.prod(orders[k + 1:])) for k in range(d)]
        R = _cabi.chain_rec(d)
        cnt = _arr(counters, 2, ctypes.c_int64)
        c = [0, 0]
        chain_twin.sample(
            strides, W, _arr(cdf, W, ctypes.c_double), _arr(rec, n * W * R, ctypes.c_double).reshape(-1, R), n,
            n_steps, step0, seed, fresh, _arr(state, M, ctypes.c_int32), _arr(total, M, ctypes.c_double),
            _arr(hit, M, ctypes.c_int32), c,
            start_cdf=_arr(start_cdf, n, ctypes.c_double) if (start_cdf.value or 0) and fresh else None,
            target=_arr(target, (n + 31) // 32, ctypes.c_uint32) if (target.value or 0) else None,
            rec_steps=_arr(rec_steps, n_rec, ctypes.c_int32) if n_rec else None,
            rec_out=_arr(rec_out, n_rec * M, ctypes.c_int32).reshape(n_rec, M) if n_rec else None)
        cnt += c
        self.launches += 1
        return 0


class _Api(object):
    def __init__(self, pkg, backend):
        self.pkg = pkg
        self.backend = backend
        self.SysDescription = pkg.SysDescription

    def DPSolver(self, sys, **kw):
        if self.backend == "model":
            kw["_test_lib"] = ChainFakeLib()
        return self.pkg.DPSolver(sys, **kw)


@pytest.fixture(scope="module", params=[pytest.param("model", id="model"),
                                        pytest.param("cuda", marks=gpu, id="cuda")])
def api(request, product):
    return _Api(product, request.param)


@pytest.fixture(scope="module")
def cuda_api(product):
    return _Api(product, "cuda")


# ---------------------------------------------------------------------------
# the cases: (solver, pol, n_steps, time_dependent, start, target)
# ---------------------------------------------------------------------------
def _ar1_golden(api):
    import workloads as wl
    return wl.storage_ar1(api).solver, golden("storage_ar1.npz")["pi_pol"]


def _sample_case(api, which):
    if which == "storage_ar1":                          # 41 x 61, W = 9
        solver, pol = _ar1_golden(api)
        n_steps, td = 50, False
    else:
        solver, pol, n_steps, td = _case(api, which)
        n_steps = {"inventory": 50, "searev_small": 60, "pv_storage": 240}[which]
    dims = solver._state_grid_shape
    # start: a distribution over the upper half of axis 0; target: levels of axis 0 that the paths
    # reach with a probability between 0.2 and 0.5 (exact values printed by the statistical test)
    start = np.zeros(dims)
    start[dims[0] // 2:] = np.random.default_rng(1).random((dims[0] - dims[0] // 2,) + dims[1:])
    target = np.zeros(dims, dtype=bool)
    target[{"inventory": slice(8, None), "storage_ar1": slice(0, 6), "searev_small": slice(0, 4),
            "pv_storage": 12}[which]] = True
    return solver, pol, n_steps, td, start, target


CASES = ["inventory", "storage_ar1", "searev_small", "pv_storage"]


def clamped_chain(solver, pol, t_k=None):
    """oracle_chain with the interpolation weights clamped to [0, 1] (NaN: the lower corner)"""
    search = oc.cell_search

    def clamped(*args):
        cell, lam = search(*args)
        return cell, np.clip(np.nan_to_num(lam, nan=0.0), 0.0, 1.0)

    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(oc, "cell_search", clamped)
        return oracle_chain(solver, pol, t_k)


def exact_moments(solver, pol, n_steps, td, mu0, target, steps):
    """mu_k (k in steps) of the clamped chain, sum_k <mu_k, g_bar> and P(reach target within n)"""
    chains = [clamped_chain(solver, pol[k], t_k=k) for k in range(n_steps)] if td else \
        [clamped_chain(solver, pol)] * n_steps
    t = target.reshape(-1)
    mu, nu = mu0.reshape(-1) / mu0.sum(), None
    nu = np.where(t, 0.0, mu)          # mass not yet absorbed in the target
    mus, cost = {0: mu}, 0.0
    for k, (P, gbar) in enumerate(chains):
        cost += float(np.dot(mu, gbar))
        mu = P.T @ mu
        nu = P.T @ nu
        nu[t] = 0.0
        mus[k + 1] = mu
    return [mus[k] for k in steps], cost, 1.0 - nu.sum()


def _z(K):
    return stats.norm.isf(stats.norm.sf(5.0) / K)


def _binom_ok(count, M, p, K):
    """both binomial tails of `count` successes out of M at probability p above sf(5)/K"""
    p = np.clip(p, 0.0, 1.0)
    lo = stats.binom.cdf(count, M, p)
    hi = stats.binom.sf(count - 1, M, p)
    return np.minimum(lo, hi) >= stats.norm.sf(5.0) / K


@pytest.mark.parametrize("which", CASES)
def test_statistics_against_the_exact_chain(api, which):
    solver, pol, n_steps, td, start, target = _sample_case(api, which)
    M = 20000
    steps = [0, 1, n_steps // 2, n_steps]
    total, info = solver.sample_paths(pol, start, n_steps, M, seed=11, target=target, record=steps,
                                      report_time=False)
    mus, cost, p_hit = exact_moments(solver, pol, n_steps, td, start, target, steps)
    n = start.size
    K = len(steps) * n + 2
    for j, k in enumerate(steps):
        counts = np.bincount(info["states"][j], minlength=n)
        ok = _binom_ok(counts, M, mus[j], K)
        assert ok.all(), (which, k, np.flatnonzero(~ok)[:5], counts[~ok][:5], M * mus[j][~ok][:5])
    se = total.std() / np.sqrt(M)
    assert abs(total.mean() - cost) <= _z(K) * se + 1e-9 * abs(cost), (which, total.mean(), cost, se)
    hits = int((info["hit_step"] >= 0).sum())
    assert _binom_ok(hits, M, p_hit, K), (which, hits / M, p_hit)
    assert np.array_equal(info["final_state"], info["states"][-1])
    h = info["hit_step"]
    assert h.min() >= -1 and h.max() <= n_steps
    assert info["nan_transitions"] == 0 and 0.0 <= info["clamped_share"] <= 1.0
    print(which, "clamped share", info["clamped_share"], "hit", hits / M, p_hit)


def test_philox_known_answer():
    """the published Philox-4x32-10 vector (Random123 kat_vectors) for counter 0, key 0"""
    c = chain_twin.philox4x32_10(0, 0, 0, 0, 0, 0)
    assert [int(v) for v in c] == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    u = chain_twin.u01(np.uint64(0xFFFFFFFF), np.uint64(0xFFFFFFFF))
    assert u == 1.0 - 2.0 ** -53 and chain_twin.u01(np.uint64(0), np.uint64(0)) == 0.0


def test_results_hold_what_the_sampler_defines(api):
    """paths from one multi-index, and from flat indices: the first recorded state is the start,
    the hit step agrees with the recorded states, the same seed gives the same paths"""
    solver, pol, n_steps, _, _, target = _sample_case(api, "inventory")
    total, info = solver.sample_paths(pol, (5,), 10, 300, seed=3, target=target, record=list(range(11)),
                                      report_time=False)
    assert info["states"].shape == (11, 300) and np.all(info["states"][0] == 5)
    inside = target.reshape(-1)[info["states"]]
    first = np.where(inside.any(axis=0), inside.argmax(axis=0), -1)
    assert np.array_equal(first, info["hit_step"])
    assert info["n_paths"] == 300 and info["n_steps"] == 10 and info["seed"] == 3
    idx = np.full(300, 5)
    total2, info2 = solver.sample_paths(pol, idx, 10, 300, seed=3, record=[10, 0, 10], report_time=False)
    assert np.array_equal(total, total2) and np.array_equal(info2["states"], info["states"][[10, 0, 10]])
    assert np.all(info2["hit_step"] == -1)
    total3, _ = solver.sample_paths(pol, idx, 10, 300, seed=4, report_time=False)
    assert not np.array_equal(total, total3)
    _, info0 = solver.sample_paths(pol, (5,), 0, 4, record=[0], report_time=False)
    assert np.all(info0["final_state"] == 5) and info0["clamped_share"] == 0.0


def test_argument_checks(api):
    solver, pol, _, _, start, target = _sample_case(api, "storage_ar1")
    dims = solver._state_grid_shape

    def run(**kw):
        args = dict(pol=pol, start=start, n_steps=3, n_paths=10, report_time=False)
        args.update(kw)
        return solver.sample_paths(**args)

    with pytest.raises(ValueError, match=r"array `pol` should be of shape"):
        run(pol=pol[..., :1])
    with pytest.raises(ValueError, match=r"array `start` should be of shape"):
        run(start=start.T)
    with pytest.raises(ValueError, match=r"array `start` should be of shape"):
        run(start=np.zeros(11, dtype=int))
    with pytest.raises(ValueError, match=r"flat indices"):
        run(start=np.full(10, start.size))
    with pytest.raises(ValueError, match=r"multi-index"):
        run(start=(0, dims[1]))
    with pytest.raises(ValueError, match=r"multi-index"):
        run(start=(0,))
    with pytest.raises(ValueError, match=r"non-negative"):
        bad = start.copy()
        bad[-1, -1] = -1e-3
        run(start=bad)
    with pytest.raises(ValueError, match=r"not all zero"):
        run(start=np.zeros(dims))
    with pytest.raises(ValueError, match=r"finite"):
        bad = start.copy()
        bad[0, 0] = np.nan
        run(start=bad)
    with pytest.raises(ValueError, match=r"array `target` should be of shape"):
        run(target=target[:-1])
    with pytest.raises(ValueError, match=r"boolean"):
        run(target=target.astype(int))
    for rec in ([4], [-1], [0, 1, 4]):
        with pytest.raises(ValueError, match=r"`record` steps must lie in \[0, n_steps\]"):
            run(record=rec)
    with pytest.raises(ValueError, match=r"integer steps"):
        run(record=[0.5])
    for m in (0, -3, 2 ** 31):
        with pytest.raises(ValueError, match=r"n_paths"):
            run(n_paths=m)
    with pytest.raises(ValueError, match=r"n_steps"):
        run(n_steps=-1)
    with pytest.raises(ValueError, match=r"seed"):
        run(seed=-1)
    # time-dependent system: the (T,) + ... policy of bellman_recursion
    tsolver, tpol, _, _, tstart, _ = _sample_case(api, "pv_storage")
    with pytest.raises(ValueError, match=r"array `pol` should be of shape"):
        tsolver.sample_paths(tpol[0], tstart, 3, 10, report_time=False)
    with pytest.raises(ValueError, match="exceeds"):
        tsolver.sample_paths(tpol[:10], tstart, 11, 10, report_time=False)


# ---------------------------------------------------------------------------
# GPU: bit-identity with the twin, launch shapes, resumed launches, config #5
# ---------------------------------------------------------------------------
def _twin_run(eng, C, n_steps, step0, seed, fresh, state, total, hit, start_cdf=None, target=None,
              rec_steps=None):
    """the twin on the device's own records (read back), on host copies of the inputs"""
    d = C.grid.d
    orders = list(C.grid.order[:d])
    strides = [int(np.prod(orders[k + 1:])) for k in range(d)]
    rec = C.rec.cpu().numpy().reshape(-1, _cabi.chain_rec(d))
    st, tot, h = state.copy(), total.copy(), hit.copy()
    cnt = [0, 0]
    rec_out = np.zeros((len(rec_steps), st.size), np.int32) if rec_steps is not None else None
    chain_twin.sample(strides, C.W, C.cdf.cpu().numpy(), rec, C.n, n_steps, step0, seed, fresh, st, tot, h, cnt,
                      start_cdf=start_cdf, target=target, rec_steps=rec_steps, rec_out=rec_out)
    return st, tot, h, cnt, rec_out


@gpu
@pytest.mark.parametrize("which", CASES)
def test_kernel_bit_identical_to_the_twin(cuda_api, which):
    solver, pol, n_steps, td, start, target = _sample_case(cuda_api, which)
    M, seed = 10000, 123456789012345
    steps = [0, n_steps // 3, n_steps]
    total, info = solver.sample_paths(pol, start, n_steps, M, seed=seed, target=target, record=steps,
                                      report_time=False)
    # the twin, instant by instant on the device's tables
    eng = solver.engine
    start_cdf = np.cumsum(start.reshape(-1))
    mask = solver._target_mask(target).view(np.uint32)
    st, tot, h = np.zeros(M, np.int32), np.zeros(M), np.zeros(M, np.int32)
    cnt, recs = [0, 0], np.zeros((len(steps), M), np.int32)
    for k in (range(n_steps) if td else [0]):
        P = eng.build_policy_tables(solver, np.asarray(pol[k] if td else pol, dtype=float),
                                    t_k=k if td else None, deterministic=True)
        C = eng.chain_tables(P)
        # the packed records against the twin's pack of the device's own planes
        d = P.grid.d
        planes = chain_twin.pack(d, P.W, P.g_per_w, P.n_states, P.cell.cpu().numpy()[:P.W * P.n_states],
                                 P.lam.cpu().numpy()[:d * P.lam_plane], P.g.cpu().numpy())
        assert np.array_equal(planes.view(np.int64), C.rec.cpu().numpy().reshape(planes.shape).view(np.int64))
        st, tot, h, c, r = _twin_run(eng, C, 1 if td else n_steps, k, seed, k == 0, st, tot, h,
                                     start_cdf=start_cdf, target=mask, rec_steps=steps)
        cnt = [cnt[0] + c[0], cnt[1] + c[1]]
        for j, s in enumerate(steps):
            if k <= s <= k + (1 if td else n_steps):
                recs[j] = r[j]
    assert np.array_equal(total.view(np.int64), tot.view(np.int64))
    assert np.array_equal(info["hit_step"], h) and np.array_equal(info["final_state"], st)
    assert np.array_equal(info["states"], recs)
    assert info["clamped_share"] == cnt[0] / (M * n_steps) and info["nan_transitions"] == cnt[1]
    print(which, "clamped share", info["clamped_share"])


@gpu
def test_launch_shapes_runs_and_resumed_launches(cuda_api):
    import torch
    solver, pol, n_steps, _, start, target = _sample_case(cuda_api, "storage_ar1")
    eng = solver.engine
    lib = eng.lib
    M, seed, n = 10000, 7, 60
    C = eng.chain_tables(eng.build_policy_tables(solver, np.asarray(pol, dtype=float), deterministic=True))
    start_cdf = eng.to_device(np.cumsum(start.reshape(-1)))
    mask = eng.to_device(solver._target_mask(target))
    rec_steps = eng.to_device(np.array([0, 20, 30, 45, 60], np.int32))

    def run(threads, split):
        lib.sdp_set_option(b"chain_threads", threads)
        state = torch.empty(M, dtype=torch.int32, device=eng.device)
        total = torch.empty(M, dtype=torch.float64, device=eng.device)
        hit = torch.empty(M, dtype=torch.int32, device=eng.device)
        cnt = torch.zeros(2, dtype=torch.int64, device=eng.device)
        rec = torch.empty(5 * M, dtype=torch.int32, device=eng.device)
        kw = dict(start_cdf=start_cdf, target=mask, rec_steps=rec_steps, rec_out=rec)
        if split:
            eng.chain_sample(C, state, total, hit, n // 2, 0, seed, True, cnt, **kw)
            eng.chain_sample(C, state, total, hit, n - n // 2, n // 2, seed, False, cnt, **kw)
        else:
            eng.chain_sample(C, state, total, hit, n, 0, seed, True, cnt, **kw)
        name = _cabi.last_kernel()
        return [t.cpu().numpy() for t in (state, total.view(torch.int64), hit, cnt, rec)], name

    try:
        ref, name = run(0, False)
        assert name.startswith("k_chain_sample<D=2>, 256 threads"), name
        for threads, split in [(0, False), (96, False), (1024, False), (0, True), (160, True)]:
            got, name = run(threads, split)
            assert str(threads or 256) in name
            for a, b in zip(ref, got):
                assert np.array_equal(a, b), (threads, split)
    finally:
        lib.sdp_set_option(b"chain_threads", 0)


@gpu
@pytest.mark.parametrize("which", CASES)
def test_unclamped_chain_matches_propagate_distribution(cuda_api, which):
    """where no transition is clamped the sampled chain is the forward operator's chain"""
    solver, pol, n_steps, td, start, target = _sample_case(cuda_api, which)
    M = 20000
    _, info = solver.sample_paths(pol, start, n_steps, M, seed=5, record=[n_steps], report_time=False)
    if info["clamped_share"] != 0.0:
        pytest.skip("%s: %.3g of the transitions are clamped" % (which, info["clamped_share"]))
    mu, _ = solver.propagate_distribution(pol, start / start.sum(), n_steps=None if td else n_steps,
                                          report_time=False)
    counts = np.bincount(info["states"][0], minlength=start.size)
    assert _binom_ok(counts, M, mu.reshape(-1), start.size).all()


@gpu
def test_config5(cuda_api):
    import workloads as wl
    prob = wl.storage_ar1_large(cuda_api)
    solver = prob.solver
    _, pol = solver.value_iteration(prob.J0, report_time=False)
    dims = solver._state_grid_shape
    start = np.zeros(dims)
    start[dims[0] // 2:, :] = 1.0
    target = np.zeros(dims, dtype=bool)
    target[0] = True
    # bit-identical to the twin, 2000 paths x 5 steps
    M, n, seed = 2000, 5, 99
    total, info = solver.sample_paths(pol, start, n, M, seed=seed, target=target, record=[0, n],
                                      report_time=False)
    eng = solver.engine
    C = eng.chain_tables(eng.build_policy_tables(solver, np.asarray(pol, dtype=float), deterministic=True))
    st, tot, h, cnt, rec = _twin_run(eng, C, n, 0, seed, True, np.zeros(M, np.int32), np.zeros(M),
                                     np.zeros(M, np.int32), start_cdf=np.cumsum(start.reshape(-1)),
                                     target=solver._target_mask(target).view(np.uint32), rec_steps=[0, n])
    assert np.array_equal(total.view(np.int64), tot.view(np.int64)) and np.array_equal(info["hit_step"], h)
    assert np.array_equal(info["states"], rec) and np.array_equal(info["final_state"], st)
    assert info["clamped_share"] == cnt[0] / (M * n) and info["nan_transitions"] == cnt[1]
    # 1e5 paths x 20 steps: the mean total cost against the clamped chain
    M, n = 100000, 20
    total, info = solver.sample_paths(pol, start, n, M, seed=1, report_time=False)
    _, cost, _ = exact_moments(solver, pol, n, False, start, target, [])
    se = total.std() / np.sqrt(M)
    print("config #5: clamped share", info["clamped_share"], "mean", total.mean(), "exact", cost, "se", se)
    assert abs(total.mean() - cost) <= _z(1) * se
