"""The table build of a sweep: what `Engine.build_sweep_tables` does, step by step.

    BuildPlan      decided ONCE per build, identically on every rank: the scan of the control boxes,
                   whether layout CF is a candidate, how the grid is cut over the ranks (slabs of
                   states, whole rows, whole columns), the measured re-cut of the slabs
    ShardBuild     the tables of THIS rank's shard for given boundaries: layout (A / B, factored or
                   dense, column-shared CF), position order, table sizes, the tabulation of the user's
                   callables with its fall-backs (batched -> per state, factored -> dense, g per
                   (x,u) -> per (x,u,w), CF -> BF), then the work list of the layout
    ChunkUpload    one flush of staged dyn/cost outputs: upload + K0 of the layout on that chunk

plus the pure-numpy planning helpers (slab cuts, work items, column order, CTA segments) and the
`SweepTables` record the sweeps read.  The device work goes through the Engine that owns the build
(uploads, the C ABI); nothing here launches on its own.

Reference behaviour the tables reproduce: stodynprog/stodynprog.py:432-463 (control grids),
:639-691 (the per-state loop whose dyn/cost calls are tabulated here).
"""
import ctypes
import os
import time
import weakref

import numpy as np

from . import _cabi
from . import tabulate as tb

# solver.column_hoist = "auto" uses layout CF (column-shared hoist) whenever it applies unless
# SDP_COLUMN_HOIST=0; "on" / "off" on the solver override it.  Measured on config #5, one B200
# (profiles/r1_column_tuning.txt): 1.21 ms per sweep against 2.83 ms for layout BF.
COLUMN_HOIST_DEFAULT = os.environ.get("SDP_COLUMN_HOIST", "1") != "0"
# solver.slab_axis = "auto": how a grid in layout CF is cut over several ranks ("auto" | "rows" |
# "columns").  By columns every rank tabulates and loads the tables of its own columns only;
# measured on config #5 (profiles/r2_shard_emulation.txt, one rank's streaming kernel): 0.179 ms
# against 0.233 ms per sweep for 1/8 of the grid, 0.61 against 0.65 ms for 1/2.  "auto" cuts
# by columns whenever layout CF applies and every rank gets at least 4 columns.
SLAB_AXIS_DEFAULT = os.environ.get("SDP_SLAB_AXIS", "auto")
# layout CF, pruning sweep: controls per group of the group summaries (sdp_column_groups_build,
# DESIGN.md section 4); 0 builds none.  A multiple of 4, at most 64.
COLUMN_GROUP_K = int(os.environ.get("SDP_COLUMN_GROUP_K", "8"))
# solver.column_pairs = "auto": layout CF with two rows per lane (3 shared-memory reads for 2
# backups instead of 4).  OFF by default: measured on config #5 (profiles/r2_emu_variants_pairs.txt)
# 1.58-1.67 ms per sweep against 1.15 ms with one row per lane.  The reads saved come back as bank
# conflicts: a half-warp's 16 lanes then span up to 32 table rows, and no placement of the rows in
# the 16 eight-byte bank pairs serves both the stride-2 pattern of the interior of the grid and the
# stride <= 1 patterns of the clipped control boxes without collisions (see DESIGN.md §4).
COLUMN_PAIRS_DEFAULT = os.environ.get("SDP_COLUMN_PAIRS", "0") != "0"


def _torch():
    import torch
    return torch


# ---------------------------------------------------------------------------
# planning helpers (host, numpy)
# ---------------------------------------------------------------------------
def partition_by_weight(weights, world):
    """Cut range(len(weights)) into `world` contiguous slabs of nearly equal
    total weight.  Returns the world+1 boundaries (monotone, first 0, last n)."""
    w = np.asarray(weights, dtype=np.float64)
    n = len(w)
    bounds = [0]
    if n == 0:
        return [0] * (world + 1)
    csum = np.cumsum(w)
    total = csum[-1]
    for r in range(1, world):
        target = total * r / world
        b = int(np.searchsorted(csum, target, side="left")) + 1
        # pick the nearer of the two candidate cuts
        if b - 1 > bounds[-1] and abs(csum[b - 2] - target) <= abs(csum[b - 1] - target):
            b -= 1
        b = min(max(b, bounds[-1]), n)
        bounds.append(b)
    bounds.append(n)
    return bounds


def rebalance_bounds(U_all, bounds, times, tolerance=1.03):
    """Re-cut contiguous slabs from measured slab times: the weight U(x)+1 of every
    state is scaled by its slab's time per unit weight (a piecewise-constant cost
    density), then the grid is cut into slabs of equal estimated time.  Returns the
    new boundaries, or None if the slabs are balanced within `tolerance` (slowest /
    mean), a time is missing, or nothing would move."""
    t = np.asarray(times, dtype=float)
    world = len(t)
    old = [int(b) for b in bounds]
    if world < 2 or not np.all(t > 0) or t.max() <= tolerance * t.mean():
        return None
    w = np.asarray(U_all, dtype=np.float64) + 1.0
    for r in range(world):
        sl = slice(old[r], old[r + 1])
        tot = w[sl].sum()
        if tot > 0:
            w[sl] *= t[r] / tot
    new = [int(b) for b in partition_by_weight(w, world)]
    return None if new == old else new


def make_items(unit_U, chunk, unit_off, per_entry, g_unit_off, g_per_entry, Upad):
    """Work-item table (SdpItem records) + first item of every unit.

    A unit (a state in layout A, a tile of 32 states in layout B) with unit_U controls is
    cut into ceil(unit_U / chunk) runs of EQUAL length (a multiple of 4, at most `chunk`):
    140 controls with chunk 128 become 72 + 68, not 128 + 12 - a short run costs a warp
    the same prologue (item, w-part, first row) as a long one.  Control u of a unit sits
    `u * per_entry` table entries after `unit_off[unit]` (g: `u * g_per_entry` after
    `g_unit_off[unit]`); `Upad` is layout A's row pitch per unit (None for layout B)."""
    unit_U = np.asarray(unit_U, dtype=np.int64)
    units = len(unit_U)
    n_it = (unit_U + chunk - 1) // chunk
    per_unit = (((unit_U + np.maximum(n_it, 1) - 1) // np.maximum(n_it, 1)) + 3) // 4 * 4
    item_begin = np.zeros(units + 1, dtype=np.int64)
    np.cumsum(n_it, out=item_begin[1:])
    n_items = int(item_begin[-1])
    st = np.repeat(np.arange(units, dtype=np.int64), n_it)
    kk = np.arange(n_items, dtype=np.int64) - item_begin[st]
    per = per_unit[st]
    items = np.zeros(n_items, dtype=_cabi.ITEM_DTYPE)
    items["u_begin"] = kk * per
    items["u_count"] = np.minimum(per, unit_U[st] - kk * per)
    items["state"] = st
    assert n_items == 0 or int(items["u_count"].min()) >= 1
    items["entry_base"] = np.asarray(unit_off)[st] + kk * per * per_entry
    items["g_base"] = np.asarray(g_unit_off)[st] + kk * per * g_per_entry
    items["Upad"] = 0 if Upad is None else np.asarray(Upad)[st]
    return items, item_begin


# Work items (warps) wanted per sweep launch.  A B200 keeps 148 SMs x 12..24 warps of these
# kernels resident, so a slab of a multi-GPU run (config #5 cut in 8: ~4 000 tiles of ~200
# controls) is only 2-3 waves of equally long items and its time is quantised by whole waves:
# measured per slab (profiles/r1_slab_chunks.txt) 0.373..0.449 ms with one item per tile,
# 0.384..0.390 ms with runs of <= 64 controls (about 9 waves) - 13 % on the slowest slab,
# which is the one the whole sweep waits for.  Runs are cut evenly (see the item table), so
# shorter runs cost nothing measurable on a grid that is already long (2.843 vs 2.853 ms).
ITEMS_TARGET = 148 * 96


def pick_item_chunk(unit_U, min_chunk, max_chunk=512, target=ITEMS_TARGET):
    """largest power-of-two-scaled chunk in [min_chunk, max_chunk] giving at least
    `target` work items for units with `unit_U` controls each"""
    unit_U = np.asarray(unit_U, dtype=np.int64)
    chunk = max_chunk
    while chunk > min_chunk and int(((unit_U + chunk - 1) // chunk).sum()) < target:
        chunk //= 2
    return max(chunk, min_chunk)


def host_threads(solver):
    """DPSolver.host_threads as a number: 1 unless asked otherwise; "auto" = the cores this
    process may run on (affinity mask, not the machine's count), at most 16"""
    v = getattr(solver, "host_threads", 1)
    if isinstance(v, str) and v.strip().lower() == "auto":
        try:
            return max(1, min(16, len(os.sched_getaffinity(0))))
        except AttributeError:
            return max(1, min(16, os.cpu_count() or 1))
    v = int(v)
    if v < 1:
        raise ValueError("host_threads must be >= 1 or 'auto'")
    return v


class _ColumnsNotApplicable(Exception):
    """the cut by columns was chosen by "auto" but layout CF turned out not to apply to the
    built tables: build_sweep_tables starts again with slabs of rows"""


class ColumnHoistRefused(Exception):
    """layout CF was demanded (column_hoist = 'on') for tables whose (x,w) part varies
    along a column of the grid"""


def pair_positions(r0, r1, pair_ok):
    """Positions of the rows [r0, r1) of a band for the two-rows-per-lane sweep: rows r, r+1 with
    pair_ok[r] share a lane (positions 2j, 2j+1), any other row gets a lane of its own with a
    padding position (-1) beside it; padded with -1 to a multiple of 64 (whole pairs of tiles).
    Returns the int64 array position -> row."""
    out = []
    r = r0
    while r < r1:
        if r + 1 < r1 and pair_ok[r]:
            out += [r, r + 1]
            r += 2
        else:
            out += [r, -1]
            r += 1
    out += [-1] * (-len(out) % 64)
    return np.asarray(out, dtype=np.int64)


def column_order(n_states, n_cols, band_rows=None, pair_ok=None):
    """Position order of layout CF for a slab of whole rows of state axis 0.

    The slab's local states are i = row*n_cols + col (C-order).  Layout CF walks them
    band by band (`band_rows`: row boundaries [0, ..., n_rows]; default one band), inside a
    band column by column, every column of a band padded to whole tiles of 32 rows.
    Returns (order, valid, band_tiles, band_tile_begin, tile_col, pos_row):
      order[p]  local state at position p (a padding position repeats the last row of
                its column in the band), valid[p] False on padding positions;
      band_tiles[b] tiles per column in band b; band_tile_begin[b] its first tile;
      tile_col[t] the column of tile t;
      pos_row   None, or - `pair_ok` given: two rows per lane, see pair_positions - per band the
                int64 array position (of every column) -> row of the band (row - r0), -1 = padding."""
    n_rows = n_states // n_cols
    assert n_rows * n_cols == n_states and n_rows >= 1
    if band_rows is None:
        band_rows = [0, n_rows]
    band_rows = [int(r) for r in band_rows]
    assert band_rows[0] == 0 and band_rows[-1] == n_rows and all(a < b for a, b in zip(band_rows, band_rows[1:]))
    cols = np.arange(n_cols, dtype=np.int64)
    orders, valids, band_tiles, band_tile_begin, tile_col, pos_row = [], [], [], [0], [], []
    for r0, r1 in zip(band_rows[:-1], band_rows[1:]):
        if pair_ok is None:
            tpc = (r1 - r0 + 31) // 32
            row = r0 + np.arange(32 * tpc, dtype=np.int64)
            valid_row = row < r1
            row = np.minimum(row, r1 - 1)
        else:
            pr = pair_positions(r0, r1, pair_ok)
            tpc = len(pr) // 32
            valid_row = pr >= 0
            # (a padding position repeats the nearest real row before it: any real state does)
            row = np.maximum.accumulate(np.where(valid_row, pr, r0))
            pos_row.append(np.where(valid_row, pr - r0, -1))
        orders.append((row[None, :] * n_cols + cols[:, None]).reshape(-1))
        valids.append(np.broadcast_to(valid_row[None, :], (n_cols, len(row))).reshape(-1))
        band_tiles.append(tpc)
        band_tile_begin.append(band_tile_begin[-1] + n_cols * tpc)
        tile_col.append(np.repeat(cols, tpc))
    return (np.concatenate(orders), np.concatenate(valids), band_tiles, band_tile_begin,
            np.concatenate(tile_col), pos_row if pair_ok is not None else None)


def item_run_ends(run_key):
    """run_end[i] = index one past the last item of the run of equal consecutive keys
    containing item i (layout CF: the items of one band and column)"""
    key = np.asarray(run_key)
    n = len(key)
    if n == 0:
        return np.zeros(0, dtype=np.int64)
    ends = np.concatenate([np.flatnonzero(key[1:] != key[:-1]) + 1, [n]]).astype(np.int64)
    return ends[np.searchsorted(ends, np.arange(n), side="right")]


def column_segments(item_u_count, n_ctas):
    """Layout CF: cut the item list (ordered by tile, hence by column) into at most
    `n_ctas` contiguous runs of equal weight, one per CTA - one CTA per SM, since the
    column table fills its shared memory - so that a CTA meets few column changes.
    Weight of an item: its controls plus a fixed cost.  Returns int64 [n_segs + 1]."""
    n_items = len(item_u_count)
    n_segs = max(1, min(int(n_ctas), n_items))
    seg = partition_by_weight(np.asarray(item_u_count, dtype=np.float64) + 2.0, n_segs)
    return np.asarray(seg, dtype=np.int64)


def column_piece_cuts(col_csum, fractions, n_ctas=0):
    """Layout CF, results handed out by pieces of columns: the column boundaries [0, ..., n_cols] of
    the pieces.  `col_csum[c]` = weight of the columns before c (n_cols + 1 values); piece k takes
    the share fractions[k] of the total weight (the last one the rest).  With n_ctas > 0 and at least
    2 * n_ctas columns a cut moves to the nearest multiple of n_ctas columns past the previous cut
    when that is within a third of the piece: every CTA then sweeps WHOLE columns of the piece
    (a CTA that starts or ends a piece in the middle of a column pays an extra column table and
    barrier, ~10 us).  Cuts that would leave an empty piece are dropped."""
    col_csum = np.asarray(col_csum, dtype=np.float64)
    n_cols = len(col_csum) - 1
    cuts, acc = [0], 0.0
    for f in fractions[:-1]:
        acc += f
        c = int(np.searchsorted(col_csum, acc * col_csum[-1], side="left"))
        if n_ctas > 0 and n_cols >= 2 * n_ctas:
            a = cuts[-1] + max(1, int(round((c - cuts[-1]) / float(n_ctas)))) * n_ctas
            if abs(a - c) * 3 <= max(c - cuts[-1], 1):
                c = a
        if cuts[-1] < c < n_cols:
            cuts.append(c)
    return cuts + [n_cols]


def column_prune_skip(g, lam, R0, R1, p, expect, best):
    """Layout CF, pruning: the skip decision of the column sweep for one control (twin of the device
    code: column_bound in the pre-pass, column_skip in the sweep; DESIGN.md section 4).  The control
    interpolates with weight `lam` between table rows R0 and R1 (W values each), `g` is its stage
    cost, `p` the W probabilities (expect = 0: W = 1 and p = [1]), `best` the lane's best value so
    far.  True: the value the sweep would compute is strictly greater than `best`.  Returns False
    wherever the sweep does not prune (p outside [0, 1], expect = 0 with W > 1, W > 9)."""
    R0, R1 = np.asarray(R0, dtype=np.float64), np.asarray(R1, dtype=np.float64)
    W = len(R0)
    pv = [float(x) for x in p] if expect else [1.0] * W
    if W > _cabi.FACTORED_MAX_W_REG or (not expect and W != 1) or not all(0.0 <= x <= 1.0 for x in pv):
        return False
    sum_p = 0.0
    for x in pv:
        sum_p += x
    with np.errstate(invalid="ignore", over="ignore"):
        m, a = np.float64(0.0), np.float64(0.0)
        for w in range(W):
            m = m + np.float64(pv[w]) * np.fmin(R0[w], R1[w])
            a = np.fmax(a, np.fmax(abs(R0[w]), abs(R1[w])))
        if np.isnan(R0).any() or np.isnan(R1).any():
            a = np.float64(np.nan)
        g = np.float64(g)
        ga = abs(g) + a
        margin = ga * np.float64(sum_p) * np.float64(2.0 ** -48) + np.float64(2.0 ** -1000)
        lb = (g * np.float64(sum_p) + m) - margin
        return bool(0.0 <= lam <= 1.0 and ga <= 2.0 ** 1000 and lb > best)


def column_group_skip(gmin, gabs, m_lo, acol, sum_p, best):
    """Layout CF, group skipping: the decision of the column sweep for one lane and one group of
    controls (twin of column_group_skip in the device code; DESIGN.md section 4).  `gmin` / `gabs`
    the least stage cost and a bound of |g| over the lane's live controls of the group, `m_lo` a
    lower bound of the row bound m(q) over their rows, `acol` the largest A(q) of the column's
    rows 0..rows-2 (NaN when one is NaN), `sum_p` the sum of the probabilities in w order, `best`
    the lane's best value so far.  The caller has checked that the group is eligible (every weight
    in [0, 1], no NaN in g, every row <= rows-2).  True: column_prune_skip holds for every member."""
    with np.errstate(invalid="ignore", over="ignore"):
        ga = np.float64(gabs) + np.float64(acol)
        margin = ga * np.float64(sum_p) * np.float64(2.0 ** -48) + np.float64(2.0 ** -1000)
        lb = (np.float64(gmin) * np.float64(sum_p) + np.float64(m_lo)) - margin
        return bool(ga <= 2.0 ** 1000 and lb > best)


def column_group_summary(g, lam, q, live, rows):
    """Layout CF, group skipping: the summary of one (item, group, lane) as the device builds it
    (k_column_groups): g, lam and the table rows q of the group's K controls of the lane, `live`
    which of them are live.  Returns (gmin, gabs, qlo, qhi): qlo = 0xffff when no control is live,
    qhi = 0xffff when the group is not eligible; gabs is rounded up to fp32."""
    g, lam = np.asarray(g, dtype=np.float64), np.asarray(lam, dtype=np.float64)
    q, live = np.asarray(q, dtype=np.int64), np.asarray(live, dtype=bool)
    if not live.any():
        return 0.0, 0.0, 0xffff, 0
    g, lam, q = g[live], lam[live], q[live]
    ok = bool(np.all((lam >= 0.0) & (lam <= 1.0)) and not np.isnan(g).any() and q.min() >= 0 and q.max() <= rows - 2)
    if not ok:
        return float(np.fmin.reduce(np.append(g, np.inf))), float("inf"), 0, 0xffff
    return float(g.min()), float_round_up(np.abs(g).max()), int(q.min()), int(q.max())


def float_round_up(x):
    """the least fp32 value >= x (inf above the largest finite fp32)"""
    with np.errstate(over="ignore"):
        f = np.float32(x)
    if np.isfinite(f) and np.float64(f) < x:
        f = np.nextafter(f, np.float32(np.inf))
    return float(f)


def window_minima(m, L):
    """Wm[q] = min m over [q, min(q+L, rows-1)) for q < rows-1 (the last row's bound is the
    sentinel and takes no part), NaN dropped as fmin does"""
    m = np.asarray(m, dtype=np.float64)
    n = len(m) - 1
    return np.array([np.fmin.reduce(m[q:min(q + L, n)]) for q in range(n)])


def group_row_bound(Wm, L, qlo, qhi):
    """the lower bound of m over [qlo, qhi] the sweep uses, from the window minima (None: the span
    exceeds 2L and the group is needed)"""
    if qhi - qlo >= 2 * L:
        return None
    return float(np.fmin(Wm[qlo], Wm[max(qlo, qhi - L + 1)]))


def build_column_groups(eng, T, K=None):
    """Layout CF: build and register the group summaries of T's u-part (sdp_column_groups_build),
    held by T.col_groups; the registration ends with release_column_groups or when T is collected.
    Every path that rewrites T.cell / T.lam / T.g goes through a table build (sdp_build_tables*),
    which also drops it."""
    K = COLUMN_GROUP_K if K is None else K
    release_column_groups(T)
    if not K or not T.column or T.pairs:
        return
    lib, nb, gid = eng.lib, ctypes.c_int64(0), ctypes.c_int64(0)
    _cabi.check(lib.sdp_column_groups_bytes(ctypes.byref(T.c_tables), K, eng.stream, ctypes.byref(nb)),
                "sdp_column_groups_bytes")
    T.col_groups = _torch().empty(max(int(nb.value), 16), dtype=_torch().uint8, device=eng.device)
    _cabi.check(lib.sdp_column_groups_build(ctypes.byref(T.grid), ctypes.byref(T.c_tables), K,
                                            eng._ptr(T.col_groups), int(nb.value), eng.stream, ctypes.byref(gid)),
                "sdp_column_groups_build")
    T.col_groups_id = int(gid.value)
    T.col_groups_fin = weakref.finalize(T, lib.sdp_column_groups_release, int(gid.value))


def release_column_groups(T):
    """end the registration of T's group summaries and free them (before the tables are rewritten)"""
    fin = getattr(T, "col_groups_fin", None)
    if fin is not None:
        fin()
    T.col_groups_fin = None
    T.col_groups = None
    T.col_groups_id = 0


def row_aligned(bounds, n_cols):
    """slab boundaries moved to the nearest multiple of n_cols (whole rows of axis 0),
    kept monotone"""
    out = [int(bounds[0])]
    for b in bounds[1:-1]:
        out.append(max(out[-1], int(round(float(b) / n_cols)) * n_cols))
    out.append(int(bounds[-1]))
    return [min(b, out[-1]) for b in out]


# ---------------------------------------------------------------------------
# the tables of a shard
# ---------------------------------------------------------------------------
class SweepTables(object):
    """Dense (cell, lam, g) tables of one slab of states, resident in HBM,
    plus the host-side control discretisation needed to turn argmin indices
    back into control values."""

    def __init__(self):
        self.grid = None           # _cabi.SdpGrid
        self.d = 0
        self.W = 1
        self.expect = 1
        self.g_per_w = 0
        self.bounds = None         # slab boundaries over ranks (world+1)
        self.state_begin = 0
        self.n_states = 0
        self.host_full = None      # HostStateTable of ALL states (replicated)
        self.cell = self.lam = self.g = self.p = None
        self.p_host = None
        self.items = self.item_begin = None
        self.part_val = self.part_idx = None
        self.J_out = self.argmin = None
        self.lam_plane = 0
        self.n_items = 0
        self.n_entries = 0
        self.n_backups_local = 0   # admissible (x,u,w) triples in this slab
        self.n_backups_total = 0
        self.c_tables = None       # _cabi.SdpTables
        self.tiled = False         # layout B (state-minor) when True
        self.u_mask = 0            # factored layouts: coordinates of the (x,u) part; 0 = dense
        self.cell_w = self.lam_w = None
        self.lam_w_plane = 0
        self.U_dev = None
        self.tabulate_mode = None
        self.setup_seconds = 0.0
        self.setup_split = None    # seconds per stage of the build, see BuildPlan.run
        self.item_chunk = 0        # controls per work item used for these tables
        self.item_begin_host = self.unit_U_host = None
        self.chunk_plan = None     # see Engine._chunk_plan
        # layout CF (column-shared hoist): BF tables over column-major tiles, see column_order()
        self.column = False
        self.n_cols = self.tiles_per_col = 0
        self.seg_begin = None      # device int64 [n_segs+1]: item range of every CTA
        self.n_segs = 0
        self.item_u_count_host = None
        self.col_table = None      # device fp64 scratch: the column tables of the current sweep
        self.col_bound = None      # device fp64 scratch: their per-row bounds (SdpTables.col_bound)
        self.col_groups = None     # device bytes: the registered group summaries (build_column_groups)
        self.col_groups_id = 0
        self.col_groups_fin = None
        self.run_end = None        # device int64 [n_items]: end of every item's (band, column) run
        self.pairs = False         # layout CF with two rows per lane (SdpTables.col_pairs)
        self.pos_row = self.work_dev = self.work_host = None
        self.item_order = None     # several bands: device int64 [n_items], items column by column (all bands)
        self.run_end_ord = None    # ... and the end of every position's column run in that order
        self.bands = None          # dict(rows, tiles, tile_begin, tile_col), see column_order
        self.band_views = None     # per band: (SdpTables view for the combine pass, first state, states)
        self.sm_count = 148
        # grid sharded by COLUMNS (layout CF, solver.slab_axis = "columns"): this rank holds the
        # columns [col_bounds[rank], col_bounds[rank+1]) of every row; local state row*n_cols + lc
        self.col_bounds = None
        self.gather_index = None   # device int64 [n_grid]: see Collective.all_gather_indexed
        self.gather_maxc = 0
        self.slab_times_ms = None  # measured per-rank sweep times (several ranks, see _measured_bounds)
        self.slab_recut = False    # True when those times moved the slab boundaries

    @property
    def algorithmic_bytes_per_backup(self):
        """4 + 8 d + 8 kappa  (SURVEY.md §8d)"""
        kappa = 1.0 if self.g_per_w else 1.0 / self.W
        return 4.0 + 8.0 * self.d + 8.0 * kappa

    @property
    def factored(self):
        return self.u_mask != 0

    @property
    def layout_name(self):
        if self.column:
            return "column_factored"
        return ("state_minor" if self.tiled else "control_minor") + ("_factored" if self.u_mask else "")

    @property
    def device_bytes(self):
        n = 0
        for t in (self.cell, self.lam, self.g, self.items, self.item_begin, self.cell_w, self.lam_w):
            if t is not None:
                n += t.numel() * t.element_size()
        return n

    @property
    def streamed_bytes_per_backup(self):
        """bytes of table the sweep kernel actually reads per admissible (x,u,w)"""
        return self.device_bytes / max(self.n_backups_local, 1)


def fill_c_tables(T):
    """the SdpTables record (include/sdp_b200.h) of a SweepTables"""
    c = _cabi.SdpTables()
    c.cell = T.cell.data_ptr()
    c.lam = T.lam.data_ptr()
    c.lam_plane = T.lam_plane
    c.g = T.g.data_ptr()
    c.g_per_w = T.g_per_w
    c.W = T.W
    c.expect = T.expect
    if T.u_mask:
        c.layout = _cabi.LAYOUT_STATE_MINOR_FACTORED if T.tiled else _cabi.LAYOUT_CONTROL_MINOR_FACTORED
        if T.column:
            c.layout = _cabi.LAYOUT_COLUMN_FACTORED
            c.n_cols, c.tiles_per_col = T.n_cols, T.tiles_per_col
            c.seg_begin, c.n_segs = T.seg_begin.data_ptr(), T.n_segs
            c.col_table = T.col_table.data_ptr()
            c.col_bound = T.col_bound.data_ptr()
            c.col_table_ready = 0
            if T.item_order is not None:
                # several bands: the whole-list launch walks the bands of a column back to back
                c.item_order = T.item_order.data_ptr()
                c.run_end = T.run_end_ord.data_ptr()
            else:
                c.run_end = T.run_end.data_ptr()
            if getattr(T, "pairs", False):
                c.col_pairs = 1
                c.pos_row = T.pos_row.data_ptr()
        c.u_mask = T.u_mask
        c.cell_w = T.cell_w.data_ptr()
        c.lam_w = T.lam_w.data_ptr()
        c.lam_w_plane = T.lam_w_plane
    else:
        c.layout = _cabi.LAYOUT_STATE_MINOR if T.tiled else _cabi.LAYOUT_CONTROL_MINOR
    c.p = T.p.data_ptr()
    c.p_host = T.p_host.ctypes.data
    c.items = T.items.data_ptr()
    c.n_items = T.n_items
    c.item_begin = T.item_begin.data_ptr()
    c.n_states = T.n_states
    c.U = T.U_dev.data_ptr()
    return c


# ---------------------------------------------------------------------------
# the build
# ---------------------------------------------------------------------------
class BuildPlan(object):
    """What a table build decides once, identically on every rank (the decisions rest on
    replicated data or are agreed through the collective).

    Solver knobs read here:
      solver.table_layout   : "auto" | "control_minor" (A) | "state_minor" (B)
      solver.table_compress : "auto" | "off" | "on"  (factored (x,u) + (x,w) tables)
      solver.tabulate       : "auto" | "per_state" | "batched"
      solver.column_hoist, solver.column_pairs, solver.slab_axis, solver.slab_balance,
      solver.host_threads
    `forced_axis` = "rows": the cut by columns chosen by "auto" was refused by the built tables.
    `for_risk`: tables for the risk sweep (sdp_sweep_risk_partials), which takes layout CF with one
    row per lane or dense layout A: where CF does not apply, the tables are dense layout A."""

    def __init__(self, eng, solver, t_k, forced_axis=None, for_risk=False):
        self.t_start = time.perf_counter()
        self.eng, self.solver, self.t_k = eng, solver, t_k
        self.for_risk = bool(for_risk)
        self.sys = sys = solver.sys
        self.state_grid = state_grid = [np.asarray(g, dtype=float) for g in solver.state_grid]
        self.d = d = len(state_grid)
        self.grid = _cabi.make_grid(state_grid)
        for ax in state_grid:
            if len(ax) < 2:
                raise ValueError("every state variable needs at least 2 grid points "
                                 "(the reference's interpolation reads out of bounds and "
                                 "divides 0/0 on a 1-point axis, SURVEY.md App. A.2)")
        self.n_grid = n_grid = int(np.prod([len(ax) for ax in state_grid]))
        # several perturbations (a TODO of the reference, stodynprog.py:666,679-683): their product
        # grid is flattened in C order into one axis of W nodes (tabulate.perturb_layout)
        self.nb_perturb = nb_perturb = len(solver.perturb_grid)
        self.W = W = tb.perturb_layout(solver.perturb_grid)[2]
        if W > 4096:
            raise ValueError("the product perturbation grid has %d nodes; at most 4096 are supported" % W)
        self.w_grid = [np.asarray(g) for g in solver.perturb_grid]
        self.coll = eng.coll
        self.world, self.rank = world, rank = eng.coll.world, eng.coll.rank
        self.dev = eng.device
        self.mode = getattr(solver, "tabulate", "auto")
        self.nb_control = nb_control = len(sys.control)
        self.compress = getattr(solver, "table_compress", "auto")
        self.keep_staging = bool(getattr(solver, "_keep_staging", False))
        self.n_host_threads = host_threads(solver)
        self.split = {}            # seconds per stage (SweepTables.setup_split)

        # pass 1: control boxes (replicated host table, needed to map argmin -> control values)
        self.eq = [n_grid * r // world for r in range(world + 1)]
        t0 = time.perf_counter()
        self.host_full, self.mine = eng._scan_boxes(solver, t_k, state_grid, n_grid, self.mode)
        self.split["scan"] = time.perf_counter() - t0
        self.U_all = self.host_full.U.astype(np.int64)
        if self.U_all.max(initial=0) >= 2 ** 31 - 4:
            raise ValueError("more than 2^31 control combinations for one state")

        # layout CF (column-shared hoist, include/sdp_b200.h): wanted by solver.column_hoist,
        # possible when the column table fits shared memory; needs slabs of whole rows of
        # state axis 0, a factored split with u_mask == 1 and a w-part that is the same for
        # all the states of a column (checked on the built tables, see ShardBuild.resolve)
        self.n_rows0 = n_rows0 = len(state_grid[0])
        self.n_cols = n_cols = n_grid // n_rows0
        self.col_mode = col_mode = getattr(solver, "column_hoist", "auto")
        if col_mode not in ("auto", "on", "off"):
            raise ValueError("column_hoist must be 'auto', 'on' or 'off'")
        col_wanted = col_mode == "on" or (col_mode == "auto" and COLUMN_HOIST_DEFAULT)
        self.col_candidate = bool(
            col_wanted and d in (2, 3) and nb_perturb >= 1 and 1 < W <= _cabi.FACTORED_MAX_W_REG
            and 8 * _cabi.column_pitch(n_rows0, W) <= _cabi.COLUMN_MAX_SMEM_BYTES
            and getattr(solver, "table_layout", "auto") in ("auto", "state_minor")
            and self.compress != "off"
            and n_rows0 >= 32 * world and nb_control <= _cabi.SDP_MAX_C)
        self.col_refused = False   # set when the built w-part turns out to vary along a column
        # layout CF with two rows per lane (SdpTables.col_pairs): solver.column_pairs / SDP_COLUMN_PAIRS
        pair_mode = getattr(solver, "column_pairs", "auto")
        if pair_mode not in ("auto", "on", "off"):
            raise ValueError("column_pairs must be 'auto', 'on' or 'off'")
        self.pairs = bool(self.col_candidate and not self.for_risk
                          and (pair_mode == "on" or (pair_mode == "auto" and COLUMN_PAIRS_DEFAULT))
                          and 8 * _cabi.column_pitch(n_rows0, W, pairs=True) <= _cabi.COLUMN_MAX_SMEM_BYTES)
        # several ranks: slabs of whole rows of axis 0 ("rows"), or - layout CF only - whole
        # columns ("columns": every rank then tabulates and loads the tables of its own columns
        # only, so the per-column costs divide by the number of ranks)
        slab_axis = getattr(solver, "slab_axis", "auto")
        if slab_axis not in ("auto", "rows", "columns"):
            raise ValueError("slab_axis must be 'auto', 'rows' or 'columns'")
        if slab_axis == "auto":
            slab_axis = SLAB_AXIS_DEFAULT
        self.axis_auto = slab_axis == "auto" or forced_axis is not None
        if forced_axis is not None:
            slab_axis = forced_axis
        elif slab_axis == "auto":
            slab_axis = "columns" if (self.col_candidate and n_cols >= 4 * world) else "rows"
        self.by_columns = world > 1 and slab_axis == "columns"
        # developer experiments (scripts/dev_shard_emulation.py): the tables of ONE column shard
        # [c0, c1) of the grid on a single rank, as a rank of a multi-GPU run would hold them
        self.col_override = getattr(solver, "_col_override", None) if world == 1 else None
        if self.col_override is not None:
            self.by_columns = True
        if self.by_columns and not (self.col_candidate and n_cols >= world):
            raise ValueError("slab_axis='columns' needs layout CF (column_hoist) and at least one "
                             "grid column per rank")

    def shard_bounds(self):
        """the cut of the grid over the ranks, balanced by admissible controls: boundaries in
        states, or (by_columns) in columns"""
        world, n_grid, n_rows0, n_cols, U_all = self.world, self.n_grid, self.n_rows0, self.n_cols, self.U_all
        if self.col_override is not None:
            return [int(self.col_override[0]), int(self.col_override[1])]
        if self.by_columns:
            # whole columns per rank, cut by the admissible controls of the columns
            col_w = (U_all + 1).reshape(n_rows0, n_cols).sum(axis=0)
            bounds = [int(b) for b in partition_by_weight(col_w, world)]
        elif world > 1 and self.col_candidate:
            # whole rows of axis 0 per rank (layout CF); a row is 1/n_rows0 of the grid
            row_w = (U_all + 1).reshape(n_rows0, n_cols).sum(axis=1)
            bounds = [int(b) * n_cols for b in partition_by_weight(row_w, world)]
        else:
            bounds = partition_by_weight(U_all + 1, world) if world > 1 else [0, n_grid]
        override = getattr(self.solver, "_slab_override", None)
        if override is not None and world == 1:
            # developer experiments (scripts/dev_slab_chunks.py): the tables of ONE slab of
            # the grid, as a rank of a multi-GPU run would hold them; only the streaming
            # kernel can be run on such tables (J_out covers the slab, not the grid)
            bounds = [int(override[0]), int(override[1])]
        return bounds

    def run(self, reuse):
        """build this rank's tables; with several ranks re-cut the slabs once by the measured
        cost of a backup in each slab and build again"""
        eng = self.eng
        T = ShardBuild(self, self.shard_bounds(), reuse).run()
        balance = getattr(self.solver, "slab_balance", "auto")
        # (layout CF cuts whole rows of axis 0 and keeps the cut by admissible controls unless
        # the measured re-cut is asked for explicitly)
        if self.world > 1 and eng._cuda and balance != "controls" and not self.by_columns and \
                (balance == "measured" or (T.n_backups_total >= eng.REBALANCE_MIN_BACKUPS and not T.column)):
            new_bounds = eng._measured_bounds(T, self.U_all)
            if new_bounds is not None and T.column:
                new_bounds = row_aligned(new_bounds, self.n_cols)
                if new_bounds == [int(b) for b in T.bounds]:
                    new_bounds = None
            if new_bounds is not None:
                T = ShardBuild(self, new_bounds, T).run()
                T.slab_recut = True
        t0 = time.perf_counter()
        eng.sync()
        self.split["device_drain"] = time.perf_counter() - t0      # uploads + K0 still in flight
        T.setup_seconds = time.perf_counter() - self.t_start
        T.setup_split = dict((k, float(v)) for k, v in self.split.items())
        return T


class ChunkUpload(object):
    """The flush of one run of staged chunks: the descriptors and the un-broadcast dyn/cost outputs
    go up in one copy, K0 of the shard's layout turns them into table entries.  `launch` can be
    called again later with other pointers (a recursion whose dynamics ignore the instant re-runs
    K0 per instant on that instant's costs, Engine.recursion_fast)."""

    def __init__(self, sb, L, g_per_w, u_mask, desc, staging):
        eng, plan, T = sb.plan.eng, sb.plan, sb.T
        self.sb, self.L, self.g_per_w, self.u_mask = sb, L, g_per_w, u_mask
        if u_mask:
            tb.check_factorable(desc, plan.d, u_mask)
        self.desc = desc
        self.desc_dev, self.stag_dev = eng.to_device_concat(desc, staging, plan.n_host_threads)
        self.n_staging = int(self.stag_dev.numel())
        self.ns = len(desc)
        self.first = L["done"]
        if sb.tiled:
            assert self.first % 32 == 0
            self.t_first = self.first // 32
            self.nt = (self.ns + 31) // 32
            self.t_off = ctypes.c_void_p(L["tile_off_dev"].data_ptr() + 8 * self.t_first)
            self.t_U = ctypes.c_void_p(L["tile_U_dev"].data_ptr() + 4 * self.t_first)
            self.t_Umax = int(L["tile_U"][self.t_first:self.t_first + self.nt].max())
        self.max_Upad = int(desc["Upad"].max()) if not sb.tiled else 0
        # (`keep`: the device arrays the launch points into)
        self.keep = (self.desc_dev, L["tile_off_dev"], L["tile_g_off_dev"], L["tile_U_dev"]) if sb.tiled \
            else (self.desc_dev,)
        self.launch(eng._ptr(self.desc_dev), eng._ptr(self.stag_dev), eng._ptr(T.g))
        L["done"] += self.ns
        # the staging tensors are freed by torch's caching allocator in stream order, so no
        # synchronisation is needed here

    def launch(self, desc_ptr, stag_ptr, g_ptr):
        """K0 on this chunk: `desc_ptr` / `stag_ptr` the chunk's descriptors and staged outputs,
        `g_ptr` the stage-cost table to fill"""
        if self.sb.tiled:
            (self._k0_state_minor_factored if self.u_mask else self._k0_state_minor)(desc_ptr, stag_ptr, g_ptr)
        else:
            (self._k0_control_minor_factored if self.u_mask else self._k0_control_minor)(desc_ptr, stag_ptr, g_ptr)

    def _k0_state_minor_factored(self, desc_ptr, stag_ptr, g_ptr):      # layouts BF and CF
        eng, plan, T, L = self.sb.plan.eng, self.sb.plan, self.sb.T, self.L
        w0 = self.t_first * plan.W * 32
        rc = eng.lib.sdp_build_tables_factored_tiled(
            ctypes.byref(plan.grid), plan.W, self.u_mask, self.ns, desc_ptr, stag_ptr,
            self.nt, self.t_off, self.t_U, self.t_Umax, eng._ptr(T.cell), eng._ptr(T.lam), L["lam_plane"],
            g_ptr, ctypes.c_void_p(T.cell_w.data_ptr() + 4 * w0),
            ctypes.c_void_p(T.lam_w.data_ptr() + 8 * w0), L["lam_w_plane"], eng.stream)
        _cabi.check(rc, "sdp_build_tables_factored_tiled")

    def _k0_state_minor(self, desc_ptr, stag_ptr, g_ptr):               # layout B
        eng, plan, T, L = self.sb.plan.eng, self.sb.plan, self.sb.T, self.L
        rc = eng.lib.sdp_build_tables_tiled(
            ctypes.byref(plan.grid), plan.W, self.g_per_w, self.ns, desc_ptr, stag_ptr,
            self.nt, self.t_off, ctypes.c_void_p(L["tile_g_off_dev"].data_ptr() + 8 * self.t_first), self.t_U,
            self.t_Umax, eng._ptr(T.cell), eng._ptr(T.lam), L["lam_plane"], g_ptr, eng.stream)
        _cabi.check(rc, "sdp_build_tables_tiled")

    def _k0_control_minor_factored(self, desc_ptr, stag_ptr, g_ptr):    # layout AF
        eng, plan, T, L = self.sb.plan.eng, self.sb.plan, self.sb.T, self.L
        w0 = self.first * plan.W
        rc = eng.lib.sdp_build_tables_factored(
            ctypes.byref(plan.grid), plan.W, self.u_mask, self.ns, desc_ptr, stag_ptr,
            eng._ptr(T.cell), eng._ptr(T.lam), L["lam_plane"], g_ptr,
            self.max_Upad, ctypes.c_void_p(T.cell_w.data_ptr() + 4 * w0),
            ctypes.c_void_p(T.lam_w.data_ptr() + 8 * w0), L["lam_w_plane"], eng.stream)
        _cabi.check(rc, "sdp_build_tables_factored")

    def _k0_control_minor(self, desc_ptr, stag_ptr, g_ptr):             # layout A
        eng, plan, T, L = self.sb.plan.eng, self.sb.plan, self.sb.T, self.L
        rc = eng.lib.sdp_build_tables(ctypes.byref(plan.grid), plan.W, self.g_per_w, self.ns,
                                      desc_ptr, stag_ptr, eng._ptr(T.cell), eng._ptr(T.lam), L["lam_plane"],
                                      g_ptr, self.max_Upad, eng.stream)
        _cabi.check(rc, "sdp_build_tables")

    def record(self):
        """what Engine.recursion_fast keeps of a flush"""
        return dict(desc=self.desc, n_staging=self.n_staging, stag_dev=self.stag_dev, launch=self.launch,
                    first=self.first, keep=self.keep)


class ShardBuild(object):
    """Tables of this rank's shard: states [bounds[rank], bounds[rank+1]) of the C-order grid, or
    (plan.by_columns) the columns [bounds[rank], bounds[rank+1]) of every row."""

    def __init__(self, plan, bounds, reuse):
        self.plan, self.bounds, self.reuse = plan, bounds, reuse
        rank, n_grid, n_rows0, n_cols = plan.rank, plan.n_grid, plan.n_rows0, plan.n_cols
        if plan.by_columns:
            c0, c1 = bounds[rank], bounds[rank + 1]
            # local state row*(c1-c0) + lc  <->  grid state row*n_cols + c0 + lc
            self.glob = (np.arange(n_rows0, dtype=np.int64)[:, None] * n_cols
                         + np.arange(c0, c1, dtype=np.int64)[None, :]).reshape(-1)
            self.sb, self.se, self.n = 0, n_grid, len(self.glob)
            self.n_cols_loc = c1 - c0
        else:
            self.sb, self.se = bounds[rank], bounds[rank + 1]
            self.n = self.se - self.sb
            self.glob = slice(self.sb, self.se)
            self.n_cols_loc = n_cols
        hf = plan.host_full
        self.host = tb.HostStateTable(self.n, plan.nb_control)
        self.host.lo, self.host.hi, self.host.npts = hf.lo[self.glob], hf.hi[self.glob], hf.npts[self.glob]
        self.U = plan.U_all[self.glob]
        self._pos = {}
        self.flushes, self.chunk_record = [], []
        self.T = None

    # -- layout ---------------------------------------------------------------
    def choose_layout(self):
        """lane <-> control (A) when states have many controls, lane <-> state (B) when there are
        many states with few controls each; factored tables when the probe state shows the
        (x,u) + (x,w) structure; layout CF when the plan wants it and the shard is whole rows or
        columns.  All ranks agree (they run the same kernels on the same layout)."""
        plan, n, U = self.plan, self.n, self.U
        solver, coll = plan.solver, plan.coll
        layout = getattr(solver, "table_layout", "auto")
        if layout == "auto":
            mean_U = float(U.mean()) if n else 0.0
            layout = "state_minor" if (n >= 32 * 1024 and mean_U <= 1024) else "control_minor"
        self.tiled = tiled = layout == "state_minor"

        # factored ("broadcast-compressed") tables when every next-state coordinate
        # depends on (x,u) only or on (x,w) only and g does not depend on w; probed on
        # the slab's state with most controls, then checked on every staged chunk
        compress, W, d = plan.compress, plan.W, plan.d
        u_mask = 0
        w_cap = _cabi.FACTORED_MAX_W_REG if tiled else _cabi.FACTORED_MAX_W_SMEM
        if (compress != "off" and n > 0 and plan.nb_perturb >= 1 and 1 < W <= w_cap and d in (2, 3)
                and plan.nb_control <= _cabi.SDP_MAX_C):
            i_probe = int(np.argmax(U))
            # (host row i_probe is grid state glob[i_probe] when the shard is whole columns)
            g_probe = int(self.glob[i_probe]) if plan.by_columns else self.sb + i_probe
            x_probe = tb.state_tuples_at(plan.state_grid, g_probe, g_probe + 1)[0]
            u_mask = tb.probe_factor_mask(plan.sys, x_probe, self.host, i_probe, plan.w_grid, plan.t_k) or 0
        if compress == "on" and not u_mask:
            raise ValueError("table_compress='on' but the system's dyn/cost do not have the "
                             "(x,u) + (x,w) structure (or d, W are outside the supported range)")
        if plan.world > 1:
            u_mask = min(coll.all_gather_object(u_mask))
        self.u_mask = u_mask
        n_cols = plan.n_cols
        column = bool(plan.col_candidate and not plan.col_refused and tiled and u_mask == 1 and n > 0
                      and (plan.by_columns or (self.sb % n_cols == 0 and self.se % n_cols == 0)))
        if plan.world > 1:
            column = bool(min(coll.all_gather_object(column)))
        if plan.by_columns and not column:
            if plan.axis_auto:
                raise _ColumnsNotApplicable()
            raise ValueError("slab_axis='columns' but layout CF does not apply to these tables")
        if plan.col_mode == "on" and not column:
            raise ValueError("column_hoist='on' but layout CF does not apply: it needs the "
                             "state-minor layout, a factored (x,u)+(x,w) split with state axis 0 "
                             "alone following the control, at most 9 perturbation nodes, a w-part "
                             "that does not depend on axis 0, and order[0]*(W|1)*8 bytes of "
                             "shared memory")
        self.column = column
        if plan.for_risk and not column:
            self.tiled, self.u_mask = False, 0       # the risk sweep's other layout: dense A

    def positions(self, col):
        """(n_eff, U_eff, host_eff, flat_eff, valid, bands): the shard's states in table order -
        C-order, or for layout CF band by band, column by column, with padding (column_order)"""
        if col not in self._pos:
            n, U, host, plan = self.n, self.U, self.host, self.plan
            if not col:
                self._pos[col] = (n, U, host, None, None, None)
            else:
                ncl = self.n_cols_loc
                bands = plan.eng._column_bands(U.reshape(n // ncl, ncl).sum(axis=1), plan.W)
                pair_ok = None
                if plan.pairs:
                    # rows that may share a lane: neighbours on axis 0 with the same control
                    # grid sizes in every column (their backups then read overlapping table
                    # rows); a speed hint only - the kernel handles any pair
                    npts_rc = host.npts.reshape(n // ncl, ncl * max(plan.nb_control, 1))
                    pair_ok = np.all(npts_rc[1:] == npts_rc[:-1], axis=1)
                order, valid, band_tiles, band_tile_begin, tile_col, pos_row = \
                    column_order(n, ncl, bands, pair_ok)
                h = tb.HostStateTable(len(order), plan.nb_control)
                h.lo, h.hi, h.npts = host.lo[order], host.hi[order], host.npts[order]
                flat = self.glob[order] if plan.by_columns else self.sb + order
                self._pos[col] = (len(order), np.where(valid, U[order], 0), h, flat, valid,
                                  dict(rows=bands, tiles=band_tiles, tile_begin=band_tile_begin,
                                       tile_col=tile_col, pos_row=pos_row))
        return self._pos[col]

    def sizes(self, u_mask, col):
        """entry offsets of the layout: dense tables have W entries per control, factored tables
        one.  Returns (n_tiles, tile_U, tile_off, n_entries, entry_off, Upad)."""
        Wf = 1 if u_mask else self.plan.W
        n, U = self.positions(col)[:2]
        if self.tiled:
            return self._sizes_state_minor(n, U, Wf, col)
        return self._sizes_control_minor(n, U, Wf)

    def _sizes_state_minor(self, n, U, Wf, col):
        """layouts B / BF / CF: tiles of 32 positions, every tile as long as its longest state"""
        n_tiles = (n + 31) // 32
        Upad_t = np.zeros(n_tiles * 32, dtype=np.int64)
        Upad_t[:n] = U
        tile_U = Upad_t.reshape(n_tiles, 32).max(axis=1)
        if col and self.plan.pairs:
            # the two tiles of a pair are swept by one warp: same number of controls
            tile_U = np.repeat(tile_U.reshape(-1, 2).max(axis=1), 2)
        tile_off = np.zeros(n_tiles + 1, dtype=np.int64)
        np.cumsum(tile_U * Wf * 32, out=tile_off[1:])
        return (n_tiles, tile_U, tile_off, int(tile_off[-1]), np.zeros(n + 1, dtype=np.int64),
                np.zeros(n, dtype=np.int64))

    @staticmethod
    def _sizes_control_minor(n, U, Wf):
        """layouts A / AF: one row per state, padded to a multiple of 4 controls"""
        Upad = (U + 3) // 4 * 4
        entry_off = np.zeros(n + 1, dtype=np.int64)
        np.cumsum(Wf * Upad, out=entry_off[1:])
        return 0, None, None, int(entry_off[-1]), entry_off, Upad

    # -- the record ------------------------------------------------------------
    def new_tables(self):
        """the SweepTables record (recycled from `reuse` when the shapes allow) with everything
        that does not depend on the tabulation: sizes, probabilities, the replicated control
        discretisation, the gather index of a cut by columns"""
        plan, reuse, bounds = self.plan, self.reuse, self.bounds
        eng = plan.eng
        self.prev_mode = reuse.tabulate_mode if reuse is not None else None
        T = reuse if (reuse is not None and reuse.W == plan.W and reuse.d == plan.d
                      and reuse.tiled == self.tiled) else SweepTables()
        self.T = T
        release_column_groups(T)       # (recycled tables: their entries are about to be rewritten)
        T.grid, T.d, T.W = plan.grid, plan.d, plan.W
        T.tiled = self.tiled
        T.expect = 1 if plan.nb_perturb >= 1 else 0
        T.bounds, T.state_begin, T.n_states = bounds, self.sb, self.n
        T.col_bounds = None
        if plan.by_columns:
            # the exchange goes by grid position, not by slab: T.bounds stays None
            T.bounds, T.state_begin, T.col_bounds = None, 0, [int(b) for b in bounds]
            if plan.col_override is None:
                n_rows0, n_cols = plan.n_rows0, plan.n_cols
                widths = np.diff(np.asarray(bounds, dtype=np.int64))
                T.gather_maxc = int(widths.max()) * n_rows0
                cols = np.arange(n_cols, dtype=np.int64)
                owner = np.searchsorted(np.asarray(bounds[1:], dtype=np.int64), cols, side="right")
                lc = cols - np.asarray(bounds, dtype=np.int64)[owner]
                rows = np.arange(n_rows0, dtype=np.int64)[:, None]
                idx = owner[None, :] * T.gather_maxc + rows * widths[owner][None, :] + lc[None, :]
                T.gather_index = eng.to_device(idx.reshape(-1))
        T.host_full = plan.host_full
        T.n_backups_local = int(self.U.sum()) * plan.W
        T.n_backups_total = int(plan.U_all.sum()) * plan.W
        # host copy of the probabilities, kept alive with the tables (SdpTables.p_host)
        T.p_host = tb.joint_proba(plan.solver.perturb_proba) if plan.nb_perturb >= 1 else np.ones(1)
        # (one packed upload for the small per-table arrays)
        small = [T.p_host]
        hf = plan.host_full
        if plan.nb_control:
            small += [hf.lo.reshape(-1), hf.hi.reshape(-1), hf.npts.astype(np.int32).reshape(-1)]
        small = eng.to_device_packed(small)
        T.p = small[0]
        # replicated control discretisation, for the argmin -> control value kernel
        T.lo_dev, T.hi_dev, T.npts_dev = (small[1], small[2], small[3]) if plan.nb_control else (None, None, None)
        T.nb_control = plan.nb_control
        T.tabulate_mode = None
        return T

    def ensure(self, name, numel, dtype):
        """(re)allocate T.<name> only when the size changes (time-dependent recursions rebuild
        same-sized tables at every instant)"""
        T = self.T
        t = getattr(T, name)
        if t is None or t.numel() != numel or t.dtype != dtype:
            setattr(T, name, None)        # release before allocating the new size
            setattr(T, name, _torch().empty(numel, dtype=dtype, device=self.plan.dev))

    # -- pass 2: tabulation ------------------------------------------------------
    def tabulate(self, g_per_w, batched, u_mask, col):
        """allocate the tables of one (g_per_w, u_mask, col) variant, evaluate dyn/cost over the
        shard and turn the staged outputs into table entries (K0), chunk by chunk.  Returns the
        variant's size record L; raises NotFactorable / GDependsOnW / BatchedMismatch."""
        plan, T = self.plan, self.T
        eng, torch = plan.eng, _torch()
        d, W, tiled = plan.d, plan.W, self.tiled
        n, U, host, flat_eff, valid, _ = self.positions(col)
        n_tiles, tile_U, tile_off, n_entries, entry_off, Upad = self.sizes(u_mask, col)
        lam_plane = (n_entries + 3) // 4 * 4
        n_u = bin(u_mask).count("1")
        L = dict(u_mask=u_mask, n_tiles=n_tiles, tile_U=tile_U, tile_off=tile_off, n_entries=n_entries,
                 entry_off=entry_off, Upad=Upad, lam_plane=lam_plane, done=0)
        self.ensure("cell", max(lam_plane, 4), torch.int32)
        self.ensure("lam", max(lam_plane, 4) * (n_u if u_mask else d), torch.float64)
        if u_mask:
            n_wp = (n_tiles * 32 if tiled else n) * W
            lam_w_plane = (n_wp + 3) // 4 * 4
            self.ensure("cell_w", max(lam_w_plane, 4), torch.int32)
            self.ensure("lam_w", max(lam_w_plane, 4) * (d - n_u), torch.float64)
        else:
            T.cell_w = T.lam_w = None
            lam_w_plane = 0
        L["lam_w_plane"] = lam_w_plane
        tile_g_off = None
        if u_mask:
            # one g per (x,u) entry, indexed like the u-part
            g_off, g_len = entry_off, n_entries
            tile_g_off = tile_off
        elif tiled:
            if g_per_w:
                tile_g_off = tile_off
            else:
                tile_g_off = np.zeros(n_tiles + 1, dtype=np.int64)
                np.cumsum(tile_U * 32, out=tile_g_off[1:])
            g_off = np.zeros(n + 1, dtype=np.int64)
            g_len = int(tile_g_off[-1])
        else:
            if g_per_w:
                g_off = entry_off
            else:
                g_off = np.zeros(n + 1, dtype=np.int64)
                np.cumsum(Upad, out=g_off[1:])
            g_len = int(g_off[-1])
        if tiled:
            L["tile_off_dev"], L["tile_g_off_dev"], L["tile_U_dev"] = eng.to_device_packed(
                [tile_off, tile_g_off, tile_U.astype(np.int32)])
        L.update(g_off=g_off, tile_g_off=tile_g_off)
        self.ensure("g", max(g_len, 4), torch.float64)
        del self.flushes[:], self.chunk_record[:]
        chunk_grids = {}

        def flush(desc, staging):
            up = ChunkUpload(self, L, g_per_w, u_mask, desc, staging)
            self.flushes.append(up.record() if plan.keep_staging else None)

        align = 32 if tiled else 1
        sb, se = self.sb, self.se
        if batched:
            # time-dependent recursion: the callables are the same at every instant, so
            # the full bit-for-bit check of the batched evaluation is made at the first
            # instant and a one-state check afterwards; unchanged control boxes reuse
            # the chunk's control grids
            tb.tabulate_states_batched(plan.sys, plan.state_grid, sb, se, host, plan.w_grid, plan.t_k,
                                       entry_off, g_off, Upad, g_per_w, flush, align=align,
                                       verify=1 if self.prev_mode == "batched" else 8,
                                       # (chunks of a column-ordered grid repeat the same rows of
                                       # control grids: kept for the duration of this build)
                                       grid_cache=eng._grid_cache if plan.t_k is not None else chunk_grids,
                                       flat_index=flat_eff, valid=valid,
                                       record=self.chunk_record if plan.keep_staging else None,
                                       threads=plan.n_host_threads)
        else:
            eq, rank = plan.eq, plan.rank
            states = plan.mine if (plan.mine is not None and (sb, se) == (eq[rank], eq[rank + 1])) else \
                tb.state_tuples(plan.state_grid, sb, se)
            if col:
                states = [states[i] for i in flat_eff - sb]      # (by_columns: sb = 0, all states)
            tb.tabulate_states(plan.sys, states, host, plan.w_grid, plan.t_k, entry_off, g_off, Upad,
                               g_per_w, flush, align=align, valid=valid)
        return L

    def resolve(self):
        """mode / layout resolution: batched evaluation is tried first in "auto" mode and
        abandoned if it fails or is not bit-identical to the reference's per-state calls on the
        sample states; factored tables are abandoned for dense ones as soon as one chunk does not
        fit the split; layout CF for BF when the built (x,w) part varies along a column.
        Returns the size record L of the variant that was built; sets T.u_mask / g_per_w / column."""
        plan, T = self.plan, self.T
        mode, compress = plan.mode, plan.compress
        u_mask, column = self.u_mask, self.column
        g_per_w = T.g_per_w if (self.reuse is T and not u_mask) else 0
        batched = mode in ("auto", "batched")
        L = None
        while L is None:
            if plan.for_risk and not (column and u_mask == 1):
                self.tiled = T.tiled = False         # (CF refused: dense layout A for the risk sweep)
                u_mask, column = 0, False
            try:
                col = column and u_mask == 1
                built = self.tabulate(g_per_w, batched, u_mask, col)
                T.tabulate_mode = "batched" if batched else "per_state"
                if col:
                    # the hoisted table is shared by a column only if the (x,w) part of its
                    # states is the same; checked bit for bit on the built tables
                    pos = self.positions(True)
                    ok = plan.eng._column_w_part_ok(T, plan.W, self.n_cols_loc, pos[5], pos[4],
                                                    built["lam_w_plane"])
                    if plan.world > 1:
                        ok = bool(min(plan.coll.all_gather_object(ok)))
                    if not ok:
                        if plan.by_columns and plan.axis_auto and plan.col_mode != "on":
                            raise _ColumnsNotApplicable()
                        if plan.col_mode == "on" or plan.by_columns:
                            raise ColumnHoistRefused("column_hoist='on' but the (x,w) part of the "
                                                     "next state depends on state axis 0")
                        plan.col_refused = True
                        column = False
                        built = None         # rebuild in C-order (layout BF)
                L = built
            except tb.NotFactorable:
                if compress == "on" or plan.world > 1:
                    # (with several ranks a silent per-rank fallback would desynchronise the layouts)
                    raise ValueError("dyn/cost outputs do not keep the (x,u) + (x,w) structure "
                                     "seen on the probe state; use solver.table_compress = 'off'")
                u_mask = 0
            except tb.GDependsOnW:
                if g_per_w:
                    raise
                if u_mask:
                    u_mask = 0
                else:
                    g_per_w = 1      # the cost depends on w: dense g table
            except tb.BatchedMismatch:
                if mode != "auto":
                    raise
                batched = False      # not bit-identical to per-state calls
            except ColumnHoistRefused as e:
                raise ValueError(str(e))
            except _ColumnsNotApplicable:
                raise
            except Exception:
                if not (batched and mode == "auto"):
                    raise
                batched = False      # callables not vectorisable over states
        T.u_mask = u_mask
        T.g_per_w = g_per_w
        T.column = bool(column and u_mask == 1)
        return L

    # -- the work list -----------------------------------------------------------
    def work_items(self, L):
        """cut the units (states of layout A, tiles of layouts B / CF) into work items, one warp
        each; layout CF adds the CTA segments and the column-by-column walking order.  Uploads the
        lists and sets the T fields the sweeps read."""
        plan, T = self.plan, self.T
        eng, torch = plan.eng, _torch()
        tiled, col, u_mask = self.tiled, T.column, T.u_mask
        T.bands = self.positions(True)[5] if col else None
        T.n_cols, T.tiles_per_col = (self.n_cols_loc, T.bands["tiles"][0]) if col else (0, 0)
        U_eff = self.positions(col)[1]
        tile_U, tile_off = L["tile_U"], L["tile_off"]
        T.n_entries, T.lam_plane, T.lam_w_plane = L["n_entries"], L["lam_plane"], L["lam_w_plane"]
        Wf = 1 if u_mask else plan.W     # table entries per control

        # work items: one warp per run of at most `item_chunk` controls
        unit_U = tile_U if tiled else self.U
        chunk = eng.item_chunk
        self.sm_count = torch.cuda.get_device_properties(plan.dev).multi_processor_count if eng._cuda else 148
        if eng.item_chunk_auto:
            # layout A walks 128 controls per warp iteration, layout B one; layout CF has one
            # CTA per SM whose 16 warps share the items of a few column pieces: several
            # rounds of items per piece keep the warps of a CTA level
            chunk = pick_item_chunk(unit_U, 128 if not tiled else 32,
                                    **({"target": self.sm_count * 16 * 48} if col else {}))
        T.item_chunk = chunk
        if col and not plan.pairs and eng.COLUMN_TAIL_FRACTION > 0 and chunk >= 32:
            # layout CF: the warps of a CTA meet at a barrier at the end of every (band, column)
            # run of tiles and wait for the one that took the last item; the last tiles of every
            # run are cut into runs of half the length, handed out last, so that the wait is
            # half an item shorter (it weighs on the short sweeps of a multi-GPU shard)
            bt, tb0 = T.bands["tiles"], T.bands["tile_begin"]
            chunk_arr = np.full(len(unit_U), chunk, dtype=np.int64)
            for b, tpc in enumerate(bt):
                tail = int(round(tpc * eng.COLUMN_TAIL_FRACTION))
                if tail > 0:
                    t_in = np.arange(tb0[b + 1] - tb0[b]) % tpc
                    chunk_arr[tb0[b]:tb0[b + 1]][t_in >= tpc - tail] = chunk // 2
            chunk = chunk_arr
        if tiled:
            per_entry = Wf * 32
            g_unit_off = tile_off if (T.g_per_w or u_mask) else L["tile_g_off"]
            # (layout CF: the Upad field of an item carries the column of its tile)
            items, item_begin = make_items(unit_U, chunk, tile_off, per_entry, g_unit_off,
                                           per_entry if (T.g_per_w or u_mask) else 32,
                                           T.bands["tile_col"] if col else None)
        else:
            items, item_begin = make_items(unit_U, chunk, L["entry_off"], 1, L["g_off"], 1, L["Upad"])
        n_items = len(items)
        T.n_items = n_items
        T.item_begin_host = item_begin
        T.unit_U_host = np.asarray(unit_U, dtype=np.int64)
        T.chunk_plan = None
        up = [items if n_items else np.zeros(1, dtype=_cabi.ITEM_DTYPE), item_begin,
              U_eff.astype(np.int32) if len(U_eff) else np.zeros(1, dtype=np.int32)]
        T.item_u_count_host = items["u_count"].copy() if col else None
        T.item_order = T.run_end_ord = T.pos_row = None
        T.pairs = bool(col and plan.pairs)
        T.work_host = None
        n_bands = 0
        if col:
            n_bands = self._column_work(items, item_begin, up)
        else:
            T.n_segs, T.seg_begin, T.run_end = 0, None, None
        up = eng.to_device_packed(up)
        T.items, T.item_begin, T.U_dev = up[0], up[1], up[2]
        if col:
            T.seg_begin, T.run_end = up[3], up[4]
            if n_bands > 1 or T.pairs:
                T.item_order, T.run_end_ord = up[5], up[6]
            T.work_dev = None
            if T.pairs:
                T.work_dev, T.pos_row = up[-2], up[-1]
            self.ensure("col_table", self.n_cols_loc * _cabi.column_pitch(plan.n_rows0, plan.W, T.pairs),
                        torch.float64)
            self.ensure("col_bound", self.n_cols_loc * plan.n_rows0 * 2, torch.float64)
        else:
            T.col_table = T.col_bound = None
        T.band_views = None

    def _column_work(self, items, item_begin, up):
        """layout CF: the WORK list (what a warp takes), its cut into one segment per CTA, the end
        of every item's run of (band, column), and - several bands - the order that walks the
        bands of a column back to back.  Appends the arrays to upload to `up`; returns the number
        of bands."""
        plan, T = self.plan, self.T
        eng, ncl = plan.eng, self.n_cols_loc
        n_items = len(items)
        T.sm_count = self.sm_count
        # items of one band and column are consecutive (tiles are ordered that way)
        n_bands = len(T.bands["tiles"])
        tile_band = np.repeat(np.arange(n_bands), np.diff(T.bands["tile_begin"]))
        st_of_item = items["state"].astype(np.int64)
        item_col = T.bands["tile_col"][st_of_item]
        # the WORK list: what a warp takes - every item, or (two rows per lane) the items of
        # the first tile of every pair, each carrying the index of the same run of controls
        # in the second tile (item.g_base; the two tiles are cut alike)
        work = np.arange(n_items, dtype=np.int64)
        if T.pairs:
            n_it = np.diff(item_begin)[st_of_item]
            first = (st_of_item % 2) == 0        # (tiles per column and band are even)
            items["g_base"] = np.where(first, work + n_it, -1)
            work = work[first]
        T.work_host = work
        w_band, w_col, w_cnt = tile_band[st_of_item][work], item_col[work], T.item_u_count_host[work]
        n_ctas = self.sm_count * eng.COLUMN_SEGS_PER_SM
        if n_bands > 1 or T.pairs:
            # the launch over the whole list (device-resident sweeps) walks the work column
            # by column, the bands of a column back to back: one table load per column
            by_col = np.argsort(w_col * n_bands + w_band, kind="stable")
            order = work[by_col]
            up.append(column_segments(w_cnt[by_col], n_ctas))
            up.append(item_run_ends(w_band * ncl + w_col))      # (natural order, per band)
            up += [order, item_run_ends(w_col[by_col])]
        else:
            up.append(column_segments(w_cnt, n_ctas))
            up.append(item_run_ends(w_band * ncl + w_col))
        T.n_segs = len(up[3]) - 1
        if T.pairs:
            up += [work, np.concatenate(T.bands["pos_row"]).astype(np.int32)]
        up[0] = items            # (g_base now holds the partners)
        return n_bands

    def finish(self):
        """result buffers and the C record"""
        plan, T, n = self.plan, self.T, self.n
        torch, dev = _torch(), plan.dev
        n_part = max(T.n_items, 1) * (32 if self.tiled else 1)
        T.part_val = torch.empty(n_part, dtype=torch.float64, device=dev)
        # (-1: no choice yet; the column sweep starts each item from the choice of the previous sweep)
        T.part_idx = torch.full((n_part,), -1, dtype=torch.int32, device=dev)
        T.J_out = torch.empty(max(n, 1), dtype=torch.float64, device=dev)
        T.argmin = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
        T.c_tables = fill_c_tables(T)
        if T.column and plan.eng._cuda:
            build_column_groups(plan.eng, T)
        # (kept for Engine.recursion_fast: one chunk, one flush, batched evaluation)
        T.build_record = None
        if plan.keep_staging and T.tabulate_mode == "batched" and len(self.flushes) == 1 \
                and len(self.chunk_record) == 1 and not T.column:
            T.build_record = dict(self.flushes[0], host=self.host, w_grid=plan.w_grid, **self.chunk_record[0])
        return T

    def run(self):
        split = self.plan.split
        t0 = time.perf_counter()
        self.choose_layout()
        self.new_tables()
        t1 = time.perf_counter()
        L = self.resolve()
        t2 = time.perf_counter()
        self.work_items(L)
        T = self.finish()
        t3 = time.perf_counter()
        split["layout"] = split.get("layout", 0.0) + (t1 - t0)
        split["tabulate_upload_k0"] = split.get("tabulate_upload_k0", 0.0) + (t2 - t1)
        split["work_list"] = split.get("work_list", 0.0) + (t3 - t2)
        return T
