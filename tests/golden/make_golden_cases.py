"""problem factories shared by make_golden.py (which needs the original stodynprog) and the
tests (which only read the committed fixtures)"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import workloads as wl  # noqa: E402


def column_cases(api, **kw):
    """the two problems of column_cases.npz: grids with >= 32 rows of state axis 0, which
    the column-shared layout (CF) takes"""
    ar1 = wl.storage_ar1(api, n_E=70, n_P=5, n_w=9, steps=(0.5, 0.1), **kw)
    sea = wl.searev(api, n_E=33, n_S=4, n_A=3, **kw)
    sea.solver.control_steps = (.05,)
    return ar1, sea


def interp_check_inputs(every=10):
    """the seeded interpolation problems of reference_checks.npz, d = 1..4: (smin, smax, orders,
    values, s) with 5 000 points drawn in and around the grid, of which every `every`-th is kept"""
    import numpy as np
    rng = np.random.default_rng(7)
    cases = []
    for d in (1, 2, 3, 4):
        orders = np.array([6, 5, 4, 3][:d], dtype=np.int64)
        smin = -rng.random(d)
        smax = smin + 1 + rng.random(d)
        vals = rng.standard_normal((3, int(np.prod(orders))))
        s = smin[:, None] + (smax - smin)[:, None] * (rng.random((d, 5000)) * 3 - 1)
        cases.append((smin, smax, orders, vals, np.ascontiguousarray(s[:, ::every])))
    return cases


def storage_ar1_check(api):
    """the 9 x 11 storage-AR1 problem of reference_checks.npz and its seeded J"""
    import numpy as np
    prob = wl.storage_ar1(api, n_E=9, n_P=11, steps=(0.01, 0.1))
    return prob, np.random.default_rng(2).standard_normal((9, 11))
