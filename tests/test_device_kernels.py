"""The small kernels around the sweeps, each against a plain reference of the same operation.

* K2 interpolation (`k_interp` behind `sdp_interp` / `sdp_interp_f32`) and the host routine
  `sdp_interp_host[_f32]` against the C restatement of the reference's Cython routine
  (oracle.oracle.interp, fp64 and fp32), bit for bit: 2-point and 4097-point axes, partial,
  single and many blocks, points outside the grid, on the nodes, at smax and one ulp either side,
  NaN / inf values; the front-ends on both sides of the host-routine threshold; refusals.
* argmin -> control values at its three device sites (`k_policy_values`, the fused tails of
  `k_combine_column` and `k_combine_column_small`) against the reference's own expression,
  `make_control_grid(lo, hi, m)[idx]`, on adversarial boxes.
* Layout CF: the column tables and the prune bound (`k_column_table`, SdpTables.col_table /
  col_bound) read back and compared with numpy in the operation order the header documents; the
  bound checked as a lower bound of the exact value of sampled controls.
* `sdp_supnorm_diff` over several grid-stride passes, `sdp_rel_shift`.

Comparisons are bit for bit; NaN positions must match, NaN payloads are not compared.  The CPU
half runs the host routine, the refusals and the vectorised control-value twin without a GPU."""
import ctypes
import fractions

import numpy as np
import pytest

from test_column_prune import _kernel_value
from test_parity import COLUMN_CASES, _Api, _adversarial, _column_case

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def lib(product):
    from stodynprog_b200 import _cabi
    return _cabi.load_library()


@pytest.fixture(scope="module")
def eng(product):
    from stodynprog_b200.engine import Engine
    return Engine()


def _same(a, b):
    """bit-identical, NaN positions equal, NaN payloads ignored"""
    a, b = np.asarray(a), np.asarray(b)
    if a.dtype != b.dtype or a.shape != b.shape:
        return False
    it = np.int32 if a.dtype == np.float32 else np.int64
    na, nb = np.isnan(a), np.isnan(b)
    return bool(np.array_equal(na, nb) and np.array_equal(a[~na].view(it), b[~nb].view(it)))


def _n_diff(a, b):
    a, b = np.asarray(a), np.asarray(b)
    it = np.int32 if a.dtype == np.float32 else np.int64
    same = (a.view(it) == b.view(it)) | (np.isnan(a) & np.isnan(b))
    return int((~same).sum())


def _vp(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _sdp_grid(smin, smax, orders):
    from stodynprog_b200 import _cabi
    g = _cabi.SdpGrid()
    g.d = len(orders)
    for k in range(min(len(orders), _cabi.SDP_MAX_D)):
        g.order[k], g.smin[k], g.smax[k] = int(orders[k]), float(smin[k]), float(smax[k])
    return g


# ---------------------------------------------------------------------------
# A. K2 interpolation
# ---------------------------------------------------------------------------
# a 2-point axis (q is always 0) and a 4097-point axis in every dimension
INTERP_ORDERS = {1: [(2,), (4097,)], 2: [(2, 4097), (7, 2)], 3: [(4097, 2, 5)], 4: [(3, 2, 4097, 2), (2, 2, 2, 2)]}
INTERP_LO = [-1.5, 0.0, 2.0, -1e3]
INTERP_HI = [2.25, 1.0, 9.0, 1e3 + 0.5]
INTERP_NS = (1, 255, 256, 257, 70001)


def _axis_pool(lo, hi, order, dtype, rng):
    """adversarial points of one axis in `dtype`: random and special points (outside the grid,
    +-3e9, +-1e300, +-inf, NaN, signed zeros, ...), every grid node, smax and one ulp either side,
    smin and one ulp below, and points whose t = sn*(order-1) truncates to order-1"""
    lo_, hi_ = dtype(lo), dtype(hi)
    inf = dtype(np.inf)
    with np.errstate(over="ignore", invalid="ignore"):
        adv = _adversarial(float(lo_), float(hi_), 4096, rng).astype(dtype)
        nodes = np.linspace(float(lo_), float(hi_), order).astype(dtype)
        span = float(hi_) - float(lo_)
        top = (float(lo_) + span * (order - 1 + rng.random(64) * 0.999) / (order - 1)).astype(dtype)
        edge = np.array([hi_, np.nextafter(hi_, inf), np.nextafter(hi_, -inf), lo_, np.nextafter(lo_, -inf)],
                        dtype=dtype)
    return np.concatenate([adv, nodes, top, edge])


def _points(lo, hi, orders, n_s, dtype, rng):
    rows = []
    for k, o in enumerate(orders):
        pool = _axis_pool(lo[k], hi[k], o, dtype, rng)
        if n_s >= len(pool):
            x = np.concatenate([pool, rng.choice(pool, n_s - len(pool))])
            rng.shuffle(x)
        else:
            x = rng.choice(pool, n_s, replace=False)
        rows.append(x)
    return np.ascontiguousarray(np.stack(rows).astype(dtype))


def _values(n_v, n_grid, dtype, rng):
    """standard normal node values; with three rows, the last one has NaN and +-inf nodes"""
    V = rng.standard_normal((n_v, n_grid)).astype(dtype)
    if n_v == 3:
        idx = rng.choice(n_grid, min(n_grid, 3 if n_grid < 100 else 6), replace=False)
        V[-1, idx[0::3]] = np.nan
        V[-1, idx[1::3]] = np.inf
        V[-1, idx[2::3]] = -np.inf
    return V


def _interp_cases(d, dtype):
    """(smin, smax, orders, values, s) over the orders of dimension d, n_v in (1, 3), n_s in
    INTERP_NS; smin / smax already rounded to `dtype` (what the fp32 kernel sees)"""
    rng = np.random.default_rng(4000 + 10 * d + (dtype == np.float32))
    lo = np.array(INTERP_LO[:d], dtype=dtype)
    hi = np.array(INTERP_HI[:d], dtype=dtype)
    for orders in INTERP_ORDERS[d]:
        n_grid = int(np.prod(orders))
        for n_v in (1, 3):
            for n_s in INTERP_NS:
                yield lo, hi, orders, _values(n_v, n_grid, dtype, rng), _points(lo, hi, orders, n_s, dtype, rng)


def _oracle_interp(smin, smax, orders, V, S):
    from oracle import oracle as oc
    with np.errstate(all="ignore"):
        return oc.interp(smin, smax, orders, V, S)


def _host_interp(lib, g, V, S):
    out = np.full((V.shape[0], S.shape[1]), np.nan, dtype=V.dtype)
    fn = lib.sdp_interp_host_f32 if V.dtype == np.float32 else lib.sdp_interp_host
    n0 = lib.sdp_launch_count()
    assert fn(ctypes.byref(g), V.shape[0], _vp(V), S.shape[1], _vp(S), _vp(out)) == 0
    assert lib.sdp_launch_count() == n0            # the host routine launches nothing
    return out


def _device_interp(eng, g, V, S):
    import torch
    from stodynprog_b200 import _cabi
    f32 = V.dtype == np.float32
    vd, sd = eng.to_device(V), eng.to_device(S)
    out = torch.full((V.shape[0], S.shape[1]), float("nan"), dtype=torch.float32 if f32 else torch.float64,
                     device=eng.device)
    fn = eng.lib.sdp_interp_f32 if f32 else eng.lib.sdp_interp
    n0 = eng.lib.sdp_launch_count()
    rc = fn(ctypes.byref(g), V.shape[0], eng._ptr(vd), S.shape[1], eng._ptr(sd), eng._ptr(out), eng.stream)
    _cabi.check(rc, "sdp_interp")
    assert eng.lib.sdp_launch_count() > n0
    return out.cpu().numpy()


@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["fp64", "fp32"])
@pytest.mark.parametrize("d", [1, 2, 3, 4])
def test_host_interp_equals_oracle(lib, d, dtype):
    """the host routine against the oracle on every case the device test uses (CPU)"""
    for smin, smax, orders, V, S in _interp_cases(d, dtype):
        want = _oracle_interp(smin, smax, orders, V, S)
        got = _host_interp(lib, _sdp_grid(smin, smax, orders), V, S)
        assert _same(got, want), (orders, V.shape, S.shape, _n_diff(got, want))


@gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["fp64", "fp32"])
@pytest.mark.parametrize("d", [1, 2, 3, 4])
def test_device_interp_equals_oracle_and_host(eng, lib, d, dtype):
    """k_interp against the oracle, and against the host routine on identical inputs"""
    for smin, smax, orders, V, S in _interp_cases(d, dtype):
        g = _sdp_grid(smin, smax, orders)
        want = _oracle_interp(smin, smax, orders, V, S)
        dev = _device_interp(eng, g, V, S)
        host = _host_interp(lib, g, V, S)
        assert _same(dev, want), (orders, V.shape, S.shape, _n_diff(dev, want))
        assert _same(dev, host), (orders, V.shape, S.shape, _n_diff(dev, host))


@pytest.mark.parametrize("fn_name", ["sdp_interp", "sdp_interp_f32", "sdp_interp_host", "sdp_interp_host_f32"])
def test_interp_refusals_launch_nothing(lib, fn_name):
    """d = 0 and 5, a 1-point axis, a grid of 2^31 points, NULL pointers: SDP_EINVAL; n_v = 0 or
    n_s = 0: SDP_OK; none of them launches a kernel (runs without a GPU: nothing reaches the device)"""
    dtype = np.float32 if fn_name.endswith("f32") else np.float64
    device = "host" not in fn_name
    fn = getattr(lib, fn_name)
    V, S, out = np.zeros((1, 8), dtype), np.zeros((2, 3), dtype), np.zeros((1, 3), dtype)

    def call(g, n_v, v, n_s, s, o):
        return fn(*([ctypes.byref(g), n_v, v, n_s, s, o] + ([None] if device else [])))
    good = _sdp_grid([0.0, 0.0], [1.0, 1.0], (2, 4))
    n0 = lib.sdp_launch_count()
    bad_grids = [_sdp_grid([], [], ()), _sdp_grid([0.0] * 4, [1.0] * 4, (2, 2, 2, 2)),
                 _sdp_grid([0.0, 0.0], [1.0, 1.0], (1, 8)), _sdp_grid([0.0, 0.0], [1.0, 1.0], (8, 1)),
                 _sdp_grid([0.0, 0.0], [1.0, 1.0], (65536, 32768)), _sdp_grid([0.0], [1.0], (2 ** 31 - 1,))]
    bad_grids[1].d = 5
    for g in bad_grids:
        assert call(g, 1, _vp(V), 3, _vp(S), _vp(out)) == -1, g.d
    assert call(good, 1, None, 3, _vp(S), _vp(out)) == -1
    assert call(good, 1, _vp(V), 3, None, _vp(out)) == -1
    assert call(good, 1, _vp(V), 3, _vp(S), None) == -1
    assert call(good, -1, _vp(V), 3, _vp(S), _vp(out)) == -1
    assert call(good, 1, _vp(V), -1, _vp(S), _vp(out)) == -1
    assert b"sdp_interp" in lib.sdp_last_error()
    assert call(good, 0, None, 3, None, None) == 0
    assert call(good, 1, None, 0, None, None) == 0
    assert lib.sdp_launch_count() == n0


@gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32], ids=["fp64", "fp32"])
def test_front_end_threshold_is_invisible(product, lib, dtype):
    """multilinear_interpolation at n_v*n_s = HOST_MAX_POINTS (host routine, no launch) and one
    point more (kernel): the same bits on the common points, and those of the oracle"""
    from stodynprog_b200 import interp as ip
    N = ip.HOST_MAX_POINTS
    rng = np.random.default_rng(77)
    orders = (9, 13)
    smin, smax = np.array([-1.0, 0.5], dtype=dtype), np.array([3.0, 2.0], dtype=dtype)
    for n_v in (1, 2):
        n_s = N // n_v
        V = _values(n_v, int(np.prod(orders)), dtype, rng)
        S = _points(smin, smax, orders, n_s + 1, dtype, rng)
        outs = []
        for m, launches in ((n_s, False), (n_s + 1, True)):
            s = np.ascontiguousarray(S[:, :m])
            n0 = lib.sdp_launch_count()
            out = product.multilinear_interpolation(smin, smax, orders, V, s)
            assert (lib.sdp_launch_count() > n0) == launches, (n_v, m)
            assert out.dtype == dtype and _same(out, _oracle_interp(smin, smax, orders, V, s))
            outs.append(out)
        assert _same(outs[0], outs[1][:, :n_s])


@gpu
def test_front_end_classes_on_the_device(product, port, lib):
    """MultilinearInterpolator(dtype=float32) and interp_on_state on more than HOST_MAX_POINTS
    points (the kernel) against the oracle and the port"""
    import workloads as wl
    from stodynprog_b200 import interp as ip
    rng = np.random.default_rng(12)
    smin, smax, orders = [0.0, -2.0], [4.0, 2.0], [11, 13]
    mi = product.MultilinearInterpolator(smin, smax, orders, dtype=np.float32)
    V = _values(3, 11 * 13, np.float32, rng)
    mi.set_values(V)
    S = _points(np.float32(smin), np.float32(smax), orders, 5000, np.float32, rng)
    n0 = lib.sdp_launch_count()
    out = mi(S)
    assert lib.sdp_launch_count() > n0 and out.dtype == np.float32
    assert _same(out, _oracle_interp(np.float32(smin), np.float32(smax), orders, V, S))
    # storage AR1: a broadcast of 61 x 50 points
    prob = wl.storage_ar1(product, n_E=11, n_P=13)
    ora = wl.storage_ar1(port, n_E=11, n_P=13)
    A = np.random.default_rng(3).standard_normal((11, 13))
    A[4, 5], A[7, 2] = np.nan, np.inf
    f, fo = prob.solver.interp_on_state(A), ora.solver.interp_on_state(A)
    x = np.linspace(-1, 11, 61).reshape(-1, 1)
    y = np.linspace(-5, 5, 50)
    assert 61 * 50 > ip.HOST_MAX_POINTS
    n0 = lib.sdp_launch_count()
    got = f(x, y)
    assert lib.sdp_launch_count() > n0 and got.shape == (61, 50)
    assert _same(got, fo(x, y))


# ---------------------------------------------------------------------------
# B. argmin -> control values
# ---------------------------------------------------------------------------
NPTS_CHOICES = np.array([1, 2, 3, 7, 4001])


def _boxes(n, nc, rng):
    """(lo, hi, npts, argmin) of n states with nc controls: random boxes and adversarial ones
    (lo == hi, signed zeros, hi < lo, a subnormal width whose step underflows to 0, bounds near
    1e308 whose width overflows, infinite and NaN bounds); argmin 0, last and random"""
    npts = rng.choice(NPTS_CHOICES, (n, nc)).astype(np.int64)
    lo = rng.uniform(-10.0, 10.0, (n, nc))
    hi = lo + rng.uniform(0.0, 5.0, (n, nc))
    kind = rng.integers(0, 12, (n, nc))
    for i, c in zip(*np.nonzero(kind >= 4)):
        k = kind[i, c]
        if k == 4:
            hi[i, c] = lo[i, c]
        elif k == 5:
            lo[i, c], hi[i, c] = [(0.0, -0.0), (-0.0, 0.0), (-0.0, -0.0), (0.0, 0.0)][rng.integers(4)]
        elif k == 6:
            lo[i, c], hi[i, c] = hi[i, c], lo[i, c]
        elif k in (7, 8):
            a = [0.0, -0.0, 1e-310, -3e-320, 2.5][rng.integers(5)]
            lo[i, c], hi[i, c] = a, a + [1e-323, -1e-323, 5e-324][rng.integers(3)]
            if a == 2.5:
                hi[i, c] = np.nextafter(a, np.inf)
            npts[i, c] = [4001, 7][rng.integers(2)]
        elif k == 9:
            lo[i, c], hi[i, c] = [(-1.5e308, 1.7e308), (1.7e308, -1.6e308), (1e308, 1.7976931348623157e308)][rng.integers(3)]
        elif k == 10:
            lo[i, c], hi[i, c] = [(np.nan, 1.0), (0.0, np.nan), (np.nan, np.nan)][rng.integers(3)]
        else:
            lo[i, c], hi[i, c] = [(-np.inf, 1.0), (0.0, np.inf), (np.inf, np.inf)][rng.integers(3)]
    # flat indices must fit int32
    while True:
        big = np.prod(npts, axis=1) >= 2 ** 31
        if not big.any():
            break
        for i in np.nonzero(big)[0]:
            npts[i, int(np.argmax(npts[i]))] = 7
    total = np.prod(npts, axis=1)
    pick = rng.integers(0, 3, n)
    argmin = np.where(pick == 0, 0, np.where(pick == 1, total - 1, (rng.random(n) * total).astype(np.int64)))
    return lo, hi, npts.astype(np.int32), argmin.astype(np.int32)


def _ref_values(lo, hi, npts, argmin):
    """the reference's expression: element idx of make_control_grid(lo, hi, m), idx from
    np.unravel_index(argmin, npts)"""
    from stodynprog_b200.tabulate import make_control_grid
    n, nc = lo.shape
    out = np.empty((n, nc))
    with np.errstate(all="ignore"):
        for i in range(n):
            ind = np.unravel_index(int(argmin[i]), tuple(int(m) for m in npts[i]))
            for c in range(nc):
                out[i, c] = make_control_grid(lo[i, c], hi[i, c], int(npts[i, c]))[ind[c]]
    return out


@pytest.mark.parametrize("nc", [1, 2, 3, 4])
def test_control_axis_values_twin_on_adversarial_boxes(nc):
    """the vectorised twin (host tabulation) against the reference's expression (CPU)"""
    from stodynprog_b200.tabulate import control_axis_values
    lo, hi, npts, argmin = _boxes(1337, nc, np.random.default_rng(500 + nc))
    want = _ref_values(lo, hi, npts, argmin)
    rem = argmin.astype(np.int64)
    got = np.empty_like(want)
    for c in range(nc - 1, -1, -1):
        idx = rem % npts[:, c]
        rem //= npts[:, c]
        with np.errstate(all="ignore"):
            got[:, c] = control_axis_values(lo[:, c], hi[:, c], npts[:, c], idx)
    assert _same(got, want), _n_diff(got, want)


def _policy_values_dev(eng, lo, hi, npts, argmin):
    import torch
    from stodynprog_b200 import _cabi
    n, nc = lo.shape
    lo_d, hi_d, np_d, am_d = (eng.to_device(a) for a in (lo, hi, npts, argmin))
    pol = torch.full((n, nc), -9.0, dtype=torch.float64, device=eng.device)
    n0 = eng.lib.sdp_launch_count()
    rc = eng.lib.sdp_policy_values(n, nc, eng._ptr(lo_d), eng._ptr(hi_d), eng._ptr(np_d), eng._ptr(am_d),
                                   eng._ptr(pol), eng.stream)
    _cabi.check(rc, "sdp_policy_values")
    assert eng.lib.sdp_launch_count() == n0 + 1
    return pol.cpu().numpy()


@gpu
@pytest.mark.parametrize("nc", [1, 2, 3, 4])
def test_policy_values_kernel(eng, nc):
    """k_policy_values on 1337 states (6 blocks, the last partial)"""
    lo, hi, npts, argmin = _boxes(1337, nc, np.random.default_rng(600 + nc))
    got = _policy_values_dev(eng, lo, hi, npts, argmin)
    want = _ref_values(lo, hi, npts, argmin)
    assert _same(got, want), _n_diff(got, want)


@pytest.fixture(scope="module")
def cf_tables(product):
    """layout CF tables of a 70 x 45 storage-AR1 grid: 3 tiles per column (the last with 6 rows),
    two column blocks of the combine (the second partial)"""
    import workloads as wl
    sv = wl.storage_ar1(_Api(product, "cuda"), n_E=70, n_P=45, n_w=3, steps=(0.5, 0.1)).solver
    sv.table_layout, sv.column_hoist, sv.column_pairs = "state_minor", "on", "off"
    T = sv.sweep_tables()
    assert T.layout_name == "column_factored" and not T.pairs and len(T.bands["tiles"]) == 1
    return sv, T


def _synthetic_partials(T, target, rng):
    """partial minima whose winner, in every tile, is one random item of the tile with index
    target[row, col] (every other item worse, random indices)"""
    tpc, n_cols = T.tiles_per_col, T.n_cols
    n_rows = T.n_states // n_cols
    ib = np.asarray(T.item_begin_host, dtype=np.int64)
    n_items = int(ib[n_cols * tpc])
    pv = 1.0 + rng.random(n_items * 32)
    pi = rng.integers(0, 2 ** 31 - 1, n_items * 32).astype(np.int32)
    for c in range(n_cols):
        for ty in range(tpc):
            k0, k1 = int(ib[c * tpc + ty]), int(ib[c * tpc + ty + 1])
            assert k1 > k0
            k = int(rng.integers(k0, k1))
            rows = np.arange(ty * 32, min(ty * 32 + 32, n_rows))
            pv[k * 32 + rows - ty * 32] = 0.25
            pi[k * 32 + rows - ty * 32] = target[rows, c]
    return pv, pi


@gpu
@pytest.mark.parametrize("beside", [0, 1], ids=["k_combine_column", "k_combine_column_small"])
@pytest.mark.parametrize("nc", [1, 2, 3, 4])
def test_fused_control_values_in_the_combine(eng, cf_tables, nc, beside):
    """sdp_sweep_finalize_cols with nc > 0, on column ranges [0, 45), [7, 38) and [13, 45): the
    argmin, J and control values of the covered states equal the reference and what
    sdp_policy_values gives for the same argmin; the other columns are untouched"""
    import torch
    from stodynprog_b200 import _cabi
    sv, T = cf_tables
    lib = eng.lib
    n_cols, tpc = T.n_cols, T.tiles_per_col
    n_rows = T.n_states // n_cols
    n = n_rows * n_cols
    rng = np.random.default_rng(700 + 10 * nc + beside)
    lo, hi, npts, argmin = _boxes(n, nc, rng)
    want = _ref_values(lo, hi, npts, argmin)
    assert _same(_policy_values_dev(eng, lo, hi, npts, argmin), want)
    pv, pi = _synthetic_partials(T, argmin.reshape(n_rows, n_cols), rng)
    pv_d, pi_d = eng.to_device(pv), eng.to_device(pi)
    lo_d, hi_d, np_d = eng.to_device(lo), eng.to_device(hi), eng.to_device(npts)
    lib.sdp_set_option(b"small_combine", 1)
    try:
        for c0, c1 in ((0, n_cols), (7, 38), (13, n_cols)):
            J = torch.full((n,), -7.0, dtype=torch.float64, device=eng.device)
            A = torch.full((n,), -5, dtype=torch.int32, device=eng.device)
            pol = torch.full((n, nc), -9.0, dtype=torch.float64, device=eng.device)
            view = _cabi.SdpTables.from_buffer_copy(T.c_tables)
            view.item_begin = T.c_tables.item_begin + 8 * c0 * tpc
            view.n_cols, view.n_states = c1 - c0, n_rows * (c1 - c0)
            rc = lib.sdp_sweep_finalize_cols(ctypes.byref(view), eng._ptr(pv_d), eng._ptr(pi_d), eng._ptr(J),
                                             eng._ptr(A), n_cols, c0, nc, eng._ptr(lo_d), eng._ptr(hi_d),
                                             eng._ptr(np_d), eng._ptr(pol), beside, eng.stream)
            _cabi.check(rc, "sdp_sweep_finalize_cols")
            J, A, pol = J.cpu().numpy(), A.cpu().numpy(), pol.cpu().numpy()
            cov = np.zeros((n_rows, n_cols), dtype=bool)
            cov[:, c0:c1] = True
            cov = cov.reshape(-1)
            assert np.array_equal(A[cov], argmin[cov]) and np.all(J[cov] == 0.25), (c0, c1)
            assert _same(pol[cov], want[cov]), (c0, c1, _n_diff(pol[cov], want[cov]))
            assert np.all(A[~cov] == -5) and np.all(J[~cov] == -7.0) and np.all(pol[~cov] == -9.0), (c0, c1)
    finally:
        lib.sdp_set_option(b"small_combine", 1)


# ---------------------------------------------------------------------------
# C. column tables and prune bound
# ---------------------------------------------------------------------------
def _cf_solver(product, which, pairs="off"):
    import workloads as wl
    if which == "config5":
        sv = wl.storage_ar1_large(_Api(product, "cuda")).solver
    else:
        sv = _column_case(_Api(product, "cuda", "state_minor", "auto", "on"), which)
    sv.table_layout, sv.column_hoist, sv.column_pairs = "state_minor", "on", pairs
    T = sv.sweep_tables()
    assert T.layout_name == "column_factored" and T.pairs == (pairs == "on")
    return sv, T


def _J_cases(shape):
    """J finite, and J with NaN, +inf and -inf on about 0.3 % of the nodes each (sparse enough
    that most table rows stay finite)"""
    rng = np.random.default_rng(31)
    J = rng.standard_normal(shape) * 10.0
    Jbad = J.copy().reshape(-1)
    k = max(1, Jbad.size // 300)
    idx = rng.choice(Jbad.size, 3 * k, replace=False)
    Jbad[idx[:k]], Jbad[idx[k:2 * k]], Jbad[idx[2 * k:]] = np.nan, np.inf, -np.inf
    return {"finite": J, "nan_inf": Jbad.reshape(shape)}


def _ref_column_tables(sv, T, J):
    """R[c, q, w]: J at axis-0 node q interpolated on the axes 1..d-1 at the w-part of lane 0 of
    column c's first tile, nested lerp in the kernel's order ((1 - l)*a + l*b, last axis innermost)"""
    c = T.c_tables
    shape = sv._state_grid_shape
    d, rows = len(shape), shape[0]
    strides = [int(np.prod(shape[k + 1:])) for k in range(d)]
    W, tpc, n_cols = c.W, c.tiles_per_col, c.n_cols
    f = ((np.arange(n_cols)[:, None] * tpc * W + np.arange(W)[None, :]) * 32)          # [c][w]
    cw = T.cell_w.cpu().numpy().astype(np.int64)[f]
    lw_all = T.lam_w.cpu().numpy()
    lw = [lw_all[j * c.lam_w_plane + f] for j in range(d - 1)]
    Jf = np.ascontiguousarray(J, dtype=np.float64).reshape(-1)

    def rec(base, k):
        if k == d:
            return Jf[base]
        a = rec(base, k + 1)
        b = rec(base + strides[k], k + 1)
        lam = lw[k - 1][None]
        return (1 - lam) * a + lam * b
    with np.errstate(all="ignore"):
        R = rec(np.arange(rows, dtype=np.int64)[:, None, None] * strides[0] + cw[None], 1)     # [q][c][w]
    return np.ascontiguousarray(R.transpose(1, 0, 2))


def _pvals(T):
    c = T.c_tables
    return [float(T.p_host[w]) if c.expect else 1.0 for w in range(c.W)]


def _ref_bound(R, p):
    """(m(q), A(q)) per column and row as the header documents: m = sum_w p_w*fmin(R[q][w],
    R[q+1][w]) from 0.0 in w order, A = max_w max(|R[q][w]|, |R[q+1][w]|) (NaN with any NaN);
    (0, NaN) for the last row"""
    n_cols, rows, W = R.shape
    R0, R1 = R[:, :-1], R[:, 1:]
    m = np.zeros((n_cols, rows - 1))
    a = np.zeros((n_cols, rows - 1))
    with np.errstate(all="ignore"):
        for w in range(W):
            m = m + np.float64(p[w]) * np.fmin(R0[..., w], R1[..., w])
            a = np.fmax(a, np.fmax(np.abs(R0[..., w]), np.abs(R1[..., w])))
    a[np.isnan(R0).any(axis=2) | np.isnan(R1).any(axis=2)] = np.nan
    out = np.empty((n_cols, rows, 2))
    out[:, :-1, 0], out[:, :-1, 1] = m, a
    out[:, -1] = (0.0, np.nan)
    return out


def _run_column_table(eng, sv, T, J, tables=None, bound=None):
    import torch
    from stodynprog_b200 import _cabi
    c = _cabi.SdpTables.from_buffer_copy(T.c_tables if tables is None else tables)
    if bound is not None:
        c.col_bound = bound
    J_dev = eng.to_device(np.ascontiguousarray(J, dtype=np.float64).reshape(-1))
    T.col_table.fill_(float("nan"))
    rc = eng.lib.sdp_column_table(ctypes.byref(T.grid), ctypes.byref(c), eng._ptr(J_dev), eng.stream)
    _cabi.check(rc, "sdp_column_table")
    torch.cuda.synchronize(eng.device)
    return T.col_table.cpu().numpy()


def _read_tables(sv, T, flat):
    from stodynprog_b200 import _cabi
    c = T.c_tables
    rows, W, P = sv._state_grid_shape[0], c.W, c.W | 1
    pitch = _cabi.column_pitch(rows, W, bool(c.col_pairs))
    q = np.arange(rows)
    off = q * P + ((q >> 1) if c.col_pairs else 0)
    return flat[:c.n_cols * pitch].reshape(c.n_cols, pitch)[:, off[:, None] + np.arange(W)[None, :]]


SENTINEL = -1234.5678


@gpu
@pytest.mark.parametrize("which", COLUMN_CASES + ["config5"])
def test_column_tables_and_bound_read_back(eng, product, which):
    """col_table and col_bound of sdp_column_table against numpy, with J finite and with NaN /
    +-inf nodes; the bound is the same bits with pruning on and off"""
    sv, T = _cf_solver(product, which)
    rows = sv._state_grid_shape[0]
    p = _pvals(T)
    lib = eng.lib
    try:
        for name, J in _J_cases(sv._state_grid_shape).items():
            R = _ref_column_tables(sv, T, J)
            want_b = _ref_bound(R, p)
            bounds = []
            for prune in (0, 1):
                lib.sdp_set_option(b"col_prune", prune)
                T.col_bound.fill_(SENTINEL)
                got = _read_tables(sv, T, _run_column_table(eng, sv, T, J))
                assert _same(got, R), (name, _n_diff(got, R))
                bounds.append(T.col_bound.cpu().numpy().copy())
            assert np.array_equal(bounds[0].view(np.int64), bounds[1].view(np.int64)), name
            b = bounds[0].reshape(T.n_cols, rows, 2)
            assert _same(b[..., 0], want_b[..., 0]), (name, "m(q)", _n_diff(b[..., 0], want_b[..., 0]))
            assert _same(b[..., 1], want_b[..., 1]), (name, "A(q)", _n_diff(b[..., 1], want_b[..., 1]))
            assert np.all(b[:, -1, 0].view(np.int64) == 0) and np.isnan(b[:, -1, 1]).all(), name
            if name == "nan_inf":
                assert np.isnan(b[:, :-1, 1]).any() and np.isfinite(b[:, :-1, 1]).any()
    finally:
        lib.sdp_set_option(b"col_prune", 1)


@gpu
def test_column_bound_untouched_where_it_does_not_apply(eng, product):
    """two rows per lane (col_pairs = 1) and a col_bound 8 bytes off 16-byte alignment: the
    pre-pass writes the tables (the swizzled ones with pairs) and leaves the bound buffer as it was"""
    import torch
    for pairs in ("on", "off"):
        sv, T = _cf_solver(product, "ar1_w3", pairs)
        J = _J_cases(sv._state_grid_shape)["nan_inf"]
        R = _ref_column_tables(sv, T, J)
        n_b = T.n_cols * sv._state_grid_shape[0] * 2
        buf = torch.full((n_b + 2,), SENTINEL, dtype=torch.float64, device=eng.device)
        ptr = buf.data_ptr() + (8 if pairs == "off" else 0)
        if pairs == "off":
            assert ptr % 16 == 8
        got = _read_tables(sv, T, _run_column_table(eng, sv, T, J, bound=ptr))
        assert _same(got, R), (pairs, _n_diff(got, R))
        assert bool((buf == SENTINEL).all()), pairs


@gpu
def test_column_bound_is_a_lower_bound(eng, product):
    """ar1_w3: for sampled (state, control) pairs with an axis-0 weight in [0, 1], the device's
    m(q) gives g*sum(p) + m(q) - margin <= the exact value of the control (fractions, from the
    table entries, g and p) and <= the value computed in the kernel's order"""
    from stodynprog_b200 import _cabi
    F = fractions.Fraction
    sv, T = _cf_solver(product, "ar1_w3")
    c = T.c_tables
    shape = sv._state_grid_shape
    rows, stride0, W = shape[0], int(np.prod(shape[1:])), c.W
    J = _J_cases(shape)["finite"]
    R = _read_tables(sv, T, _run_column_table(eng, sv, T, J))
    B = T.col_bound.cpu().numpy().reshape(c.n_cols, rows, 2)
    p = _pvals(T)
    sum_p = 0.0
    for x in p:
        sum_p += x
    items = T.items.cpu().numpy().view(np.uint8)[:c.n_items * _cabi.ITEM_DTYPE.itemsize].view(_cabi.ITEM_DTYPE)
    cell, lam, g = T.cell.cpu().numpy(), T.lam.cpu().numpy(), T.g.cpu().numpy()
    U = T.U_dev.cpu().numpy()
    rng = np.random.default_rng(41)
    n_checked = 0
    for it in items[rng.choice(len(items), min(len(items), 300), replace=False)]:
        cnt, ub, eb, tix, col = (int(it[k]) for k in ("u_count", "u_begin", "entry_base", "state", "Upad"))
        for lane in range(32):
            n_ok = max(0, min(cnt, int(U[tix * 32 + lane]) - ub))
            for j in range(n_ok):
                e = eb + j * 32 + lane
                q, l, gv = int(cell[e]) // stride0, float(lam[e]), float(g[e])
                assert int(cell[e]) % stride0 == 0
                if not (0.0 <= l <= 1.0) or q + 1 >= rows:
                    continue
                m, a = B[col, q]
                ga = abs(gv) + a
                margin = ga * sum_p * 2.0 ** -48 + 2.0 ** -1000
                lb = (gv * sum_p + m) - margin
                R0, R1 = R[col, q], R[col, q + 1]
                v = _kernel_value(gv, l, R0, R1, p, c.expect)
                exact = sum(F(p[w]) * (F(gv) + (1 - F(l)) * F(float(R0[w])) + F(l) * F(float(R1[w])))
                            for w in range(W))
                assert F(float(lb)) <= exact and lb <= v, (col, q, l, gv, lb, v)
                n_checked += 1
    assert n_checked > 1000, n_checked


# ---------------------------------------------------------------------------
# D. sup-norm of the update, relative shift
# ---------------------------------------------------------------------------
def _supnorm(eng, a, b, out0=7.0):
    import torch
    from stodynprog_b200 import _cabi
    out = torch.full((1,), out0, dtype=torch.float64, device=eng.device)
    ad, bd = eng.to_device(a), eng.to_device(b)
    rc = eng.lib.sdp_supnorm_diff(eng._ptr(ad), eng._ptr(bd), a.size, eng._ptr(out), eng.stream)
    _cabi.check(rc, "sdp_supnorm_diff")
    return out.cpu().numpy()[0]


def _ref_supnorm(a, b):
    with np.errstate(invalid="ignore"):
        d = np.abs(a - b)
    d = d[~np.isnan(d)]
    return max(0.0, float(d.max())) if d.size else 0.0


@gpu
@pytest.mark.parametrize("n", [303103, 303104, 303105, 2000000])
def test_supnorm_grid_stride_passes(eng, n):
    """148*8 blocks of 256 threads = 303 104 per pass: the maximum in the last pass, +-inf,
    inf - inf = NaN (ignored), all NaN -> 0, -0.0"""
    rng = np.random.default_rng(n)
    a, b = rng.standard_normal(n), rng.standard_normal(n)
    last = (n - 1) // 303104 * 303104
    i = int(rng.integers(last, n))
    a[i], b[i] = 50.0, -50.0
    a[::1001] = np.nan
    got = _supnorm(eng, a, b)
    assert got == _ref_supnorm(a, b) == 100.0
    a2 = a.copy()
    j = i - 1 if i > 0 else 1                         # (next to the maximum)
    a2[j], b[j] = np.inf, np.inf                      # inf - inf: NaN, ignored
    assert _supnorm(eng, a2, b) == 100.0
    a2[i] = -np.inf
    assert _supnorm(eng, a2, b) == np.inf
    assert _supnorm(eng, np.full(n, np.nan), b) == 0.0
    z = _supnorm(eng, np.full(n, -0.0), np.zeros(n))
    assert z == 0.0 and np.signbit(z) == False      # noqa: E712


@gpu
def test_supnorm_empty_writes_zero(eng):
    import torch
    from stodynprog_b200 import _cabi
    out = torch.full((1,), 3.0, dtype=torch.float64, device=eng.device)
    n0 = eng.lib.sdp_launch_count()
    _cabi.check(eng.lib.sdp_supnorm_diff(None, None, 0, eng._ptr(out), eng.stream), "sdp_supnorm_diff")
    assert out.cpu().numpy()[0] == 0.0 and eng.lib.sdp_launch_count() == n0


@gpu
@pytest.mark.parametrize("where", ["first", "middle", "last"])
@pytest.mark.parametrize("at", ["finite", "nan", "inf", "-inf"])
def test_rel_shift(eng, where, at):
    """J - J[ref] in place and J[ref] in ref_out, against numpy, bit for bit"""
    import torch
    from stodynprog_b200 import _cabi
    n = 1000
    rng = np.random.default_rng(5)
    J = rng.standard_normal(n) * 100.0
    J[17], J[400] = np.inf, np.nan
    r = {"first": 0, "middle": n // 2, "last": n - 1}[where]
    J[r] = {"finite": J[r], "nan": np.nan, "inf": np.inf, "-inf": -np.inf}[at]
    Jd = eng.to_device(J)
    ref = torch.full((1,), 5.0, dtype=torch.float64, device=eng.device)
    rc = eng.lib.sdp_rel_shift(eng._ptr(Jd), n, r, eng._ptr(ref), eng.stream)
    _cabi.check(rc, "sdp_rel_shift")
    with np.errstate(invalid="ignore"):
        want = J - J[r]
    assert _same(ref.cpu().numpy(), J[r:r + 1])
    assert _same(Jd.cpu().numpy(), want)


def test_rel_shift_refusals(lib):
    n0 = lib.sdp_launch_count()
    buf = np.zeros(4)
    for n, r in ((4, 4), (4, -1), (0, 0)):
        assert lib.sdp_rel_shift(_vp(buf), n, r, _vp(buf), None) == -1
    assert lib.sdp_rel_shift(None, 4, 0, _vp(buf), None) == -1
    assert lib.sdp_rel_shift(_vp(buf), 4, 0, None, None) == -1
    assert lib.sdp_launch_count() == n0
