"""Generate the golden fixtures of tests/golden/ from the UNMODIFIED reference.

Run in the build container only (needs /root/reference):
    python tests/golden/make_golden.py [--searev-full]

The reference is imported from where it lies through oracle/ref_loader.py
(environment shims only, no source change) with its Cython routine compiled by
oracle/build_ref.py.  Problem definitions come from
tests/workloads.py, instantiated against the reference's own
SysDescription / DPSolver classes.  Outputs (.npz, compressed) are committed;
the GPU box has no /root/reference and only reads the fixtures.

Fixtures and the reference code path that produced them:
  interp_kat.npz     multilinear_interpolation (pyx:17-49), d = 1..4, incl. adversarial points
  inventory.npz      config #1, 6 x value_iteration (stodynprog.py:466-534)
  pv_storage.npz     config #2, bellman_recursion T=240 (:536-591)
  storage_ar1.npz    config #3, 3 x value_iteration from 0, eval_policy(50, rel_dp),
                     policy_iteration(pol_ini, 50, 4, rel_dp=True) (:693-812)
  searev_small.npz   config #4 callables on a 7x11x11 grid, control step .01: value_iteration x2,
                     policy_iteration(pol_lin, 30, 2, rel_dp=True)
  column_cases.npz   grids with >= 32 rows of state axis 0, which the column-shared layout (CF)
                     takes: storage-AR1 on 70 x 5 (control step 0.5): 3 x value_iteration from 0,
                     one from a random J, policy_iteration(pol_ini, 10, 2, rel_dp=True);
                     SEAREV on 33 x 4 x 3 (control step .05): 2 x value_iteration
  searev_full.npz    config #4 as shipped: policy_iteration(pol_lin, 1000, 5, rel_dp=True)
                     (== examples/20 .../storage control/pol_E10_grid3161_iter5.npy), ~15 min
  reference_checks.npz  (--reference-checks) the original's side of three cross-checks of
                     tests/test_oracle.py: multilinear_interpolation on the seeded points of
                     make_golden_cases.interp_check_inputs; value_iteration + eval_policy(5, rel_dp)
                     on the seeded 9 x 11 storage-AR1 J; the two columns of examples/01
                     .../pv_prod.csv.  The committed file holds the oracle's results on these
                     inputs (every tenth interpolation point): up to commit 3e0e2a7 the three
                     checks ran live against the reference and matched it exactly (CPU suite:
                     243 passed, 4 skipped), and neither the oracle nor the inputs changed since.
                     This option rewrites it from the reference itself.
"""
import contextlib
import io
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle.ref_loader import load_reference, load_reference_cython  # noqa: E402
import workloads as wl  # noqa: E402
sys.path.insert(0, HERE)
from make_golden_cases import column_cases, interp_check_inputs, storage_ar1_check  # noqa: E402


def quiet(fn, *a, **k):
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        out = fn(*a, **k)
    return out, buf.getvalue()


def ref_costs(text):
    return np.array([float(l.split(':')[1]) for l in text.splitlines() if 'ref policy cost' in l])


def save(name, **arrays):
    path = os.path.join(HERE, name)
    np.savez_compressed(path, **arrays)
    print('wrote %s (%.1f kB)' % (name, os.path.getsize(path) / 1e3))


def adversarial(lo, hi, n, rng):
    """coordinates in, on and far outside [lo, hi] (SURVEY.md App. A.3)"""
    span = hi - lo
    x = lo + span * (rng.random(n) * 1.6 - 0.3)           # 30 % outside on each side
    special = np.array([lo, hi, np.nextafter(hi, lo), np.nextafter(lo, hi), lo - 0.5 * span,
                        hi + 7.3 * span, 3e9, -3e9, 1e300, -1e300, 1e6, np.inf, -np.inf, np.nan,
                        0.0, -0.0, 5e-324])
    x[:len(special)] = special
    rng.shuffle(x)
    return x


def make_interp_kat(ref):
    cy = load_reference_cython()
    rng = np.random.default_rng(20131)
    out = {}
    shapes = {1: (7,), 2: (5, 9), 3: (4, 6, 5), 4: (3, 4, 5, 3)}
    for d, orders in shapes.items():
        smin = np.array([-1.0, 0.5, 2.0, -3.0][:d])
        smax = smin + np.array([2.0, 1.25, 3.0, 0.7][:d])
        n_grid = int(np.prod(orders))
        values = np.ascontiguousarray(rng.standard_normal((2, n_grid)))
        n_s = 400
        s = np.ascontiguousarray(np.stack([adversarial(smin[k], smax[k], n_s, rng) for k in range(d)]))
        with np.errstate(all='ignore'):
            res = cy.multilinear_interpolation(smin, smax, np.array(orders, dtype=np.int64), values, s)
        out['d%d_smin' % d] = smin
        out['d%d_smax' % d] = smax
        out['d%d_orders' % d] = np.array(orders, dtype=np.int64)
        out['d%d_values' % d] = values
        out['d%d_s' % d] = s
        out['d%d_out' % d] = np.asarray(res)
        # fp32 branch of the fused type
        res32 = cy.multilinear_interpolation(smin.astype(np.float32), smax.astype(np.float32),
                                             np.array(orders, dtype=np.int64),
                                             values.astype(np.float32),
                                             np.ascontiguousarray(s.astype(np.float32)))
        out['d%d_out_f32' % d] = np.asarray(res32)
    save('interp_kat.npz', **out)


def make_inventory(ref):
    prob = wl.inventory(ref)
    J = prob.J0
    Js, pols = [], []
    for k in range(6):
        (J, u), _ = quiet(prob.solver.value_iteration, J)
        Js.append(J.copy())
        pols.append(u.copy())
    save('inventory.npz', J=np.array(Js), pol=np.array(pols))


def make_pv(ref):
    prob = wl.pv_storage(ref)
    t0 = time.time()
    (J, pol), _ = quiet(prob.solver.bellman_recursion, prob.horizon, prob.J_fin)
    print('pv_storage reference: %.1f s' % (time.time() - t0))
    save('pv_storage.npz', J=J, pol=pol, backups=np.array(wl.backups_per_sweep(prob.solver, 0)))


def make_storage_ar1(ref):
    prob = wl.storage_ar1(ref)
    sv = prob.solver
    out = {}
    J = prob.J0
    for k in range(3):
        t0 = time.time()
        (J, u), _ = quiet(sv.value_iteration, J)
        print('storage_ar1 sweep %d: %.1f s' % (k, time.time() - t0))
        out['vi_J%d' % k] = J.copy()
        out['vi_pol%d' % k] = u.copy()
    pol_ini = prob.initial_policy()
    (Je, Jref_hist), _ = quiet(sv.eval_policy, pol_ini, 50, rel_dp=True, J_ref_full=True)
    out['pol_ini'] = pol_ini
    out['ev_J'] = Je
    out['ev_Jref_hist'] = Jref_hist
    ((Jd, Jr), pol), text = quiet(sv.policy_iteration, pol_ini, 50, 4, rel_dp=True)
    out['pi_J'] = Jd
    out['pi_Jref'] = np.array(Jr)
    out['pi_pol'] = pol
    out['pi_ref_costs'] = ref_costs(text)
    print('storage_ar1 ref costs:', out['pi_ref_costs'])
    dims = np.array([sv.control_grids(x)[1] for x in __import__('itertools').product(*sv.state_grid)])
    out['control_dims'] = dims
    save('storage_ar1.npz', **out)


def searev_small(api, **kw):
    prob = wl.searev(api, n_E=7, n_S=11, n_A=11, **kw)
    prob.solver.control_steps = (.01,)
    return prob


def make_searev_small(ref):
    prob = searev_small(ref)
    sv = prob.solver
    out = {}
    J = prob.J0
    for k in range(2):
        (J, u), _ = quiet(sv.value_iteration, J)
        out['vi_J%d' % k] = J.copy()
        out['vi_pol%d' % k] = u.copy()
    pol0 = prob.initial_policy()
    ((Jd, Jr), pol), text = quiet(sv.policy_iteration, pol0, 30, 2, rel_dp=True)
    out['pi_J'] = Jd
    out['pi_Jref'] = np.array(Jr)
    out['pi_pol'] = pol
    out['pi_ref_costs'] = ref_costs(text)
    save('searev_small.npz', **out)


def make_searev_full(ref):
    prob = wl.searev(ref)
    sv = prob.solver
    pol0 = prob.initial_policy()
    t0 = time.time()
    ((Jd, Jr), pol), text = quiet(sv.policy_iteration, pol0, 1000, 5, rel_dp=True)
    print('searev full policy_iteration: %.0f s' % (time.time() - t0))
    costs = ref_costs(text)
    print('ref costs', costs)
    shipped = os.path.join(os.environ.get('STODYNPROG_REFERENCE', '/root/reference'), 'examples',
                           '20 Searev storage control', 'storage control',
                           'pol_E10_grid3161_iter5.npy')
    same = None
    if os.path.exists(shipped):
        same = bool(np.array_equal(np.load(shipped), pol))
        print('bit-identical to the shipped pol_E10_grid3161_iter5.npy:', same)
    save('searev_full.npz', pi_J=Jd, pi_Jref=np.array(Jr), pi_pol=pol, pi_ref_costs=costs,
         matches_shipped_npy=np.array(same))


def make_column_cases(ref):
    ar1, sea = column_cases(ref)
    out = {}
    sv = ar1.solver
    J = ar1.J0
    for k in range(3):
        (J, u), _ = quiet(sv.value_iteration, J)
        out['ar1_vi_J%d' % k] = J.copy()
        out['ar1_vi_pol%d' % k] = u.copy()
    J_rand = np.random.default_rng(70).standard_normal(sv._state_grid_shape)
    (J, u), _ = quiet(sv.value_iteration, J_rand)
    out['ar1_J_rand'], out['ar1_vr_J'], out['ar1_vr_pol'] = J_rand, J, u
    pol_ini = ar1.initial_policy()
    ((Jd, Jr), pol), text = quiet(sv.policy_iteration, pol_ini, 10, 2, rel_dp=True)
    out['ar1_pi_J'], out['ar1_pi_Jref'], out['ar1_pi_pol'] = Jd, np.array(Jr), pol
    out['ar1_pi_ref_costs'] = ref_costs(text)
    sv = sea.solver
    J = sea.J0
    for k in range(2):
        (J, u), _ = quiet(sv.value_iteration, J)
        out['sea_vi_J%d' % k] = J.copy()
        out['sea_vi_pol%d' % k] = u.copy()
    save('column_cases.npz', **out)


def make_reference_checks(ref):
    from oracle.ref_loader import REF_ROOT
    cy = load_reference_cython()
    out = {}
    for d, (smin, smax, orders, vals, s) in enumerate(interp_check_inputs(), 1):
        out['interp_d%d' % d] = np.asarray(cy.multilinear_interpolation(smin, smax, orders, vals, s))
    prob, J = storage_ar1_check(ref)
    (out['vi_J'], out['vi_pol']), _ = quiet(prob.solver.value_iteration, J)
    (out['ev_J'], ev_ref), _ = quiet(prob.solver.eval_policy, out['vi_pol'], 5, rel_dp=True)
    out['ev_Jref'] = np.array(ev_ref)
    csv = os.path.join(REF_ROOT, 'examples', '01 Deterministic storage control', 'pv_prod.csv')
    out['pv_t'], out['pv_P'] = np.loadtxt(csv, skiprows=1, delimiter=',').T
    save('reference_checks.npz', **out)


if __name__ == '__main__':
    ref = load_reference()
    assert ref is not None, 'the reference is not available here'
    if '--searev-full' in sys.argv:
        make_searev_full(ref)
    elif '--reference-checks' in sys.argv:
        make_reference_checks(ref)
    elif '--column-cases' in sys.argv:
        make_column_cases(ref)
    else:
        make_column_cases(ref)
        make_interp_kat(ref)
        make_inventory(ref)
        make_pv(ref)
        make_storage_ar1(ref)
        make_searev_small(ref)
