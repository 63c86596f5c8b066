"""bench.py's command line and --dump-outputs files (no GPU needed)"""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT


def test_dump_outputs_whole_arrays(tmp_path):
    import bench
    J = np.random.default_rng(0).standard_normal((50, 20))
    pol = np.arange(50 * 3, dtype=np.float32).reshape(50, 3)
    bench.write_outputs(str(tmp_path), {"J": J, "pol": pol})
    a, b = np.load(tmp_path / "J.npy"), np.load(tmp_path / "pol.npy")
    assert a.dtype == b.dtype == np.float64
    assert np.array_equal(a, J) and np.array_equal(b, pol)


def test_dump_outputs_sample_is_capped_and_fixed(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 24000)
    n = 3000                             # 72 000 bytes of float64 in all
    J = np.arange(n, dtype=np.float64)
    pol = np.stack([J, -J], axis=1)
    for d in ("a", "b"):
        bench.write_outputs(str(tmp_path / d), {"J": J, "pol": pol})
    files = [tmp_path / d / f for d in ("a", "b") for f in ("J.npy", "pol.npy")]
    a, b = np.load(files[0]), np.load(files[1])
    assert a.nbytes + b.nbytes <= 24000 and 0 < a.size < n and np.all(np.diff(a) > 0)
    assert np.array_equal(b[:, 0], a) and np.array_equal(b[:, 1], -a)     # the same rows
    assert np.array_equal(np.load(files[2]), a) and np.array_equal(np.load(files[3]), b)


@pytest.mark.parametrize("layout,column", [("state_minor", "on"), ("control_minor", "auto")])
def test_dump_is_the_last_timed_sweep(product, layout, column):
    """after the loop of bench.time_sweeps (intermediate sweeps without argmin), the dumped
    (J, pol) are what value_iteration returns from the last sweep's input (numpy model of
    the library)"""
    import bench
    import workloads as wl
    from fake_lib import FakeLib
    sv = wl.storage_ar1(product, n_E=70, n_P=5, steps=(0.5, 0.1), _test_lib=FakeLib()).solver
    sv.table_layout, sv.column_hoist = layout, column
    T = sv.sweep_tables()
    eng = sv.engine
    n = 70 * 5
    J_prev, J_new = eng.J_pair(n)
    eng.begin_call(n)
    eng.upload_J(np.random.default_rng(5).standard_normal(n), J_prev)
    K = 3
    for k in range(K):
        J_in = J_prev.clone()
        eng.sweep(T, J_prev, J_new, defer_wait=True, want_argmin=(k == K - 1))
        J_prev, J_new = J_new, J_prev
    eng.flush_exchange()
    J_last, pol_last = bench.last_sweep_results(eng, T, J_prev.clone())
    J_want, pol_want = sv.value_iteration(J_in.numpy().reshape(70, 5), report_time=False)
    assert np.array_equal(J_last.view(np.int64), J_want.reshape(-1).view(np.int64))
    assert np.array_equal(pol_last, pol_want.reshape(n, -1))


def test_steps_must_be_positive():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"],
                         capture_output=True, text=True)
    assert res.returncode == 2 and "--steps" in res.stderr
