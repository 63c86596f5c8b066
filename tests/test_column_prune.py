"""Layout CF, pruning (SdpTables.col_bound, option "col_prune"): the column sweep skips the
controls whose per-row lower bound, less a rounding margin, is already worse than the lane's best
value.  The results must be those of the full sweep, bit for bit.

CPU: the skip decision (tablebuild.column_prune_skip, twin of the device code) against the value
computed in the kernel's exact operation order, and the ABI mirror.  GPU: pruning on against off
on every column case and on config #5, over several sweeps (the seeds of the previous sweep are
live), with NaN / inf in J, for every launch shape, with exact ties everywhere and with garbage
in the seed buffer."""
import ctypes
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from test_parity import COLUMN_CASES, _Api, _column_case, _same_bits

gpu = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _kernel_value(g, lam, R0, R1, p, expect):
    """the value of one control as the column sweep computes it: oml = 1 - lam, the two
    products, their sum, + g, * p_w, summed in w order from 0.0 (numpy fp64, no FMA)"""
    oml = np.float64(1.0) - np.float64(lam)
    acc = np.float64(0.0)
    for w in range(len(R0)):
        v = oml * np.float64(R0[w]) + np.float64(lam) * np.float64(R1[w])
        jg = np.float64(g) + v
        acc = acc + jg * np.float64(p[w]) if expect else jg
    return acc


def _cases(rng):
    """(g, lam, R0, R1, p, expect, best): seeded random and adversarial inputs"""
    from stodynprog_b200.tablebuild import column_prune_skip
    specials = [0.0, -0.0, 1.0, -1.0, 1e300, -1e300, 1e-310, np.inf, -np.inf, np.nan, 2.0 ** 1000]
    lams = [0.0, 1.0, 0.5, np.nextafter(0.0, -1.0), np.nextafter(1.0, 2.0), np.nextafter(1.0, 0.0),
            5e-324, 1.0 / 3.0]
    for _ in range(6000):
        W = int(rng.choice([1, 2, 5, 9]))
        expect = bool(rng.random() < 0.8) or W > 1
        if expect:
            p = rng.random(W)
            p = p / p.sum()
            if rng.random() < 0.1:
                p[rng.integers(W)] = 0.0
        else:
            p = np.ones(1)
        scale = 10.0 ** rng.integers(-300, 300) if rng.random() < 0.2 else 1.0
        R0 = rng.standard_normal(W) * scale
        R1 = R0 + rng.standard_normal(W) * scale * 10.0 ** rng.integers(-16, 1)
        if rng.random() < 0.2:
            R1 = R0.copy()                       # flat table rows
        if rng.random() < 0.05:
            R0[rng.integers(W)] = rng.choice(specials)
        g = rng.standard_normal() * (10.0 ** rng.integers(-3, 4))
        if rng.random() < 0.03:
            g = rng.choice(specials)
        lam = rng.choice(lams) if rng.random() < 0.3 else rng.random()
        v = _kernel_value(g, lam, R0, R1, p, expect)
        # the best so far: at, just below / above the bound and the value (ties at 1 ulp)
        m = sum(np.float64(p[w] if expect else 1.0) * min(R0[w], R1[w]) for w in range(W))
        lb = np.float64(g) * np.float64(sum(p) if expect else 1.0) + m
        for best in (v, np.nextafter(v, -np.inf), np.nextafter(v, np.inf), lb, np.nextafter(lb, -np.inf),
                     lb - abs(lb) * 1e-15, v - abs(v) * 1e-13 - 1e-300, lb - 1.0, np.inf, np.nan):
            yield g, lam, R0, R1, p, expect, np.float64(best), column_prune_skip


def test_skip_decision_is_exact():
    """whenever the twin says "skip", the value the kernel would compute is strictly greater than
    the best so far (never a tie, never a NaN): the control is neither the minimum nor the argmin"""
    rng = np.random.default_rng(20261020)
    n = n_skip = 0
    with np.errstate(all="ignore"):
        for g, lam, R0, R1, p, expect, best, skip in _cases(rng):
            n += 1
            if skip(g, lam, R0, R1, p, expect, best):
                n_skip += 1
                v = _kernel_value(g, lam, R0, R1, p, expect)
                assert not np.isnan(v) and v > best, (g, lam, R0, R1, p, expect, best, v)
    assert n_skip > n // 10          # the test is not vacuous


def test_skip_decision_refuses():
    """no skip outside the conditions of the bound: ties, lam outside [0, 1], NaN / inf in R or g,
    a best of +inf or NaN, p outside [0, 1], expect = 0 with W > 1"""
    from stodynprog_b200.tablebuild import column_prune_skip as skip
    R0, R1, p = np.array([1.0, 2.0]), np.array([3.0, 4.0]), np.array([0.5, 0.5])
    assert skip(0.0, 0.5, R0, R1, p, True, 0.0)
    v = _kernel_value(0.0, 0.0, R0, R1, p, True)
    assert not skip(0.0, 0.0, R0, R1, p, True, v)                   # a tie
    assert not skip(0.0, np.nextafter(0.0, -1.0), R0, R1, p, True, 0.0)
    assert not skip(0.0, np.nextafter(1.0, 2.0), R0, R1, p, True, 0.0)
    assert not skip(0.0, np.nan, R0, R1, p, True, 0.0)
    for bad in (np.nan, np.inf, -np.inf):
        assert not skip(0.0, 0.5, np.array([1.0, bad]), R1, p, True, 0.0)
        assert not skip(bad, 0.5, R0, R1, p, True, 0.0)
    assert not skip(0.0, 0.5, R0, R1, p, True, np.inf)
    assert not skip(0.0, 0.5, R0, R1, p, True, np.nan)
    assert not skip(0.0, 0.5, R0, R1, np.array([1.5, -0.5]), True, 0.0)
    assert not skip(0.0, 0.5, R0, R1, p, False, 0.0)
    assert skip(0.0, 0.5, R0[:1], R1[:1], [7.0], False, 0.0)       # deterministic: p ignored, = 1


def test_abi_mirrors_col_bound(tmp_path):
    """SdpTables.col_bound (last field) and SDP_ABI_VERSION 10 in the header and in _cabi"""
    from stodynprog_b200 import _cabi
    hdr = open(os.path.join(ROOT, "include", "sdp_b200.h")).read()
    assert int(re.search(r"#define SDP_ABI_VERSION (\d+)", hdr).group(1)) == _cabi.SDP_ABI_VERSION == 10
    T = _cabi.SdpTables
    assert T._fields_[-1] == ("col_bound", ctypes.c_void_p)
    assert "sdp_col_prune_counts" in _cabi.SIGNATURES
    cc = shutil.which("cc") or shutil.which("gcc")
    if cc is None:
        pytest.skip("no C compiler")
    src = tmp_path / "off.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "sdp_b200.h"\n'
                   'int main(void){printf("%zu %zu\\n", offsetof(SdpTables, col_bound), sizeof(SdpTables));return 0;}\n')
    exe = tmp_path / "off"
    subprocess.check_call([cc, "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    off, size = map(int, subprocess.check_output([str(exe)]).split())
    assert (off, size) == (T.col_bound.offset, ctypes.sizeof(T))


def test_tables_carry_the_bound_and_fresh_seeds(product):
    """the CF tables own a [n_cols][rows][2] bound buffer and start with no seed (-1)"""
    sv = _column_case(_Api(product, "model", "state_minor", "auto", "on"), "ar1_w3")
    sv.column_hoist = "on"
    T = sv.sweep_tables()
    assert T.layout_name == "column_factored"
    rows = sv._state_grid_shape[0]
    assert T.col_bound.numel() == T.n_cols * rows * 2 and T.c_tables.col_bound == T.col_bound.data_ptr()
    assert bool((T.part_idx == -1).all())


# ---------------------------------------------------------------------------
# GPU: pruning on against off
# ---------------------------------------------------------------------------
def _pair(product, which):
    ref = _column_case(_Api(product, "cuda", "state_minor", "auto", "on"), which)
    col = _column_case(_Api(product, "cuda", "state_minor", "auto", "on"), which)
    for sv in (ref, col):
        sv.column_hoist, sv.column_pairs = "on", "off"
    return ref, col


def _vi(sv, J, prune):
    sv.engine.lib.sdp_set_option(b"col_prune", prune)
    try:
        return sv.value_iteration(J, report_time=False)
    finally:
        sv.engine.lib.sdp_set_option(b"col_prune", 1)


def _check_sweeps(ref, col, J0, n_sweeps, inject=True):
    """value_iteration with pruning off (ref) and on (col), each on its own cached tables so
    that the seeds of the pruning side are those of its own previous sweep"""
    for sweep in range(n_sweeps):
        Jr, polr = _vi(ref, J0, 0)
        Jc, polc = _vi(col, J0, 1)
        assert col.last_tables.layout_name == "column_factored" and not col.last_tables.pairs
        assert _same_bits(Jr, Jc), sweep
        assert np.array_equal(polr, polc, equal_nan=True), sweep
        J0 = Jr.copy()
        if inject and sweep == 2:
            J0.reshape(-1)[::7] = np.nan
            J0.reshape(-1)[3::11] = np.inf
    return J0


@gpu
@pytest.mark.parametrize("which", COLUMN_CASES)
def test_prune_is_bit_identical(product, which):
    ref, col = _pair(product, which)
    J0 = np.random.default_rng(11).standard_normal(ref._state_grid_shape)
    J0 = _check_sweeps(ref, col, J0, 5)
    # CTA size, controls per iteration, prefetch depth, table copy and item hand-out
    lib = col.engine.lib
    try:
        Jr, polr = _vi(ref, J0, 0)
        for threads, ub, pf, pre in ((128, 1, 1, 1), (256, 2, 1, 0), (512, 1, 2, 0), (96, 2, 2, 2),
                                     (640, 2, 1, 2), (768, 1, 2, 0), (704, 1, 1, 2), (768, 2, 1, 3),
                                     (640, 1, 2, 3), (64, 2, 2, 3)):
            lib.sdp_set_option(b"col_threads", threads)
            lib.sdp_set_option(b"col_ub", ub)
            lib.sdp_set_option(b"col_pf", pf)
            lib.sdp_set_option(b"col_prepass", pre)
            lib.sdp_set_option(b"col_dynamic", (threads // 32) % 2)
            for _ in range(2):                  # (the second sweep starts from live seeds)
                J2, pol2 = _vi(col, J0, 1)
                assert _same_bits(Jr, J2), (threads, ub, pf, pre)
                assert np.array_equal(polr, pol2, equal_nan=True), (threads, ub, pf, pre)
    finally:
        lib.sdp_set_option(b"col_threads", 0)
        lib.sdp_set_option(b"col_ub", 2)
        lib.sdp_set_option(b"col_pf", 2)
        lib.sdp_set_option(b"col_prepass", 3)
        lib.sdp_set_option(b"col_dynamic", 1)


@gpu
def test_prune_with_ties_everywhere(product):
    """J constant along axis 0: every control of a state interpolates between equal table rows,
    so whole runs of controls tie exactly; the argmin is still the lowest index"""
    ref, col = _pair(product, "ar1_w9")
    dims = ref._state_grid_shape
    J0 = np.broadcast_to(np.random.default_rng(5).standard_normal((1,) + dims[1:]), dims).copy()
    for _ in range(4):
        Jr, polr = _vi(ref, J0, 0)
        Jc, polc = _vi(col, J0, 1)
        assert _same_bits(Jr, Jc) and np.array_equal(polr, polc, equal_nan=True)
    T = col.last_tables
    eng = col.engine
    # the device-resident sweep: argmin indices themselves, pruning on and off
    out = {}
    for prune in (0, 1, 1):
        eng.lib.sdp_set_option(b"col_prune", prune)
        J_prev, J_new = eng.J_pair(int(np.prod(dims)))
        eng.begin_call(int(np.prod(dims)))
        eng.upload_J(J0, J_prev)
        eng.sweep(T, J_prev, J_new)
        import torch
        torch.cuda.synchronize()
        out.setdefault(prune, []).append(T.argmin.cpu().numpy().copy())
    eng.lib.sdp_set_option(b"col_prune", 1)
    assert all(np.array_equal(out[0][0], a) for a in out[1])


@gpu
def test_prune_config5(product):
    """config #5 (2000 x 500 states, W = 9) over 4 device-resident sweeps: J and argmin bit for
    bit, pruning on against off, and the pruning sweep actually skips"""
    import torch
    import workloads as wl
    sv = wl.storage_ar1_large(_Api(product, "cuda")).solver
    T = sv.sweep_tables()
    assert T.layout_name == "column_factored"
    eng, lib = sv.engine, sv.engine.lib
    n = int(np.prod(sv._state_grid_shape))
    J0 = np.random.default_rng(0).standard_normal(sv._state_grid_shape)
    res = {}
    try:
        for prune in (0, 1):
            lib.sdp_set_option(b"col_prune", prune)
            lib.sdp_set_option(b"col_prune_stats", 1)
            T.part_idx.fill_(-1)
            J_prev, J_new = eng.J_pair(n)
            eng.begin_call(n)
            eng.upload_J(J0, J_prev)
            seq = []
            for _ in range(4):
                eng.sweep(T, J_prev, J_new)
                J_prev, J_new = J_new, J_prev
                torch.cuda.synchronize()
                seq.append((J_prev.clone().cpu().numpy(), T.argmin.cpu().numpy().copy()))
            steps, skipped = ctypes.c_int64(), ctypes.c_int64()
            assert lib.sdp_col_prune_counts(ctypes.byref(steps), ctypes.byref(skipped)) == 0
            res[prune] = (seq, steps.value, skipped.value)
    finally:
        lib.sdp_set_option(b"col_prune", 1)
        lib.sdp_set_option(b"col_prune_stats", 0)
    for (Ja, Aa), (Jb, Ab) in zip(res[0][0], res[1][0]):
        assert np.array_equal(Ja.view(np.int64), Jb.view(np.int64)) and np.array_equal(Aa, Ab)
    assert res[0][1] == 0 and res[1][1] > 0 and 0 < res[1][2] <= res[1][1]


@gpu
def test_prune_seeds_are_well_defined(product):
    """the first sweep after a table build (no seeds), a sweep after a build of tables of another
    shape, and a sweep over garbage in the seed buffer give the results of the full sweep"""
    ref, col = _pair(product, "ar1_w5")
    J0 = np.random.default_rng(7).standard_normal(ref._state_grid_shape)
    Jr, polr = _vi(ref, J0, 0)
    Jc, polc = _vi(col, J0, 1)                      # first sweep: part_idx = -1
    assert _same_bits(Jr, Jc) and np.array_equal(polr, polc, equal_nan=True)
    other = _column_case(_Api(product, "cuda", "state_minor", "auto", "on"), "searev")
    other.column_hoist, other.column_pairs = "on", "off"
    _vi(other, np.zeros(other._state_grid_shape), 1)
    T = col.last_tables
    rng = np.random.default_rng(8)
    for fill in ("valid", "garbage"):
        import torch
        n = T.part_idx.numel()
        if fill == "valid":
            vals = rng.integers(0, 64, n)
        else:
            vals = rng.integers(-2 ** 31, 2 ** 31 - 1, n)
        T.part_idx.copy_(torch.from_numpy(vals.astype(np.int32)))
        Jc, polc = _vi(col, J0, 1)
        assert _same_bits(Jr, Jc) and np.array_equal(polr, polc, equal_nan=True), fill
