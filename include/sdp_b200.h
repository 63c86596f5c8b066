/*
 * sdp_b200.h - C ABI of the B200-native Bellman backward-induction engine.
 *
 * This is the drop-in boundary of the hot path of pierre-haessig/stodynprog:
 * plain pointers and sizes, no torch / numpy / C++ types.  All pointers named
 * "device" are CUDA device pointers owned by the caller (the Python host code
 * owns them through torch tensors and passes `tensor.data_ptr()`); `stream` is a
 * `cudaStream_t` passed as `void*` (NULL = legacy default stream).
 *
 * Conventions (SURVEY.md §8b):
 *   - every entry point returns 0 on success, a negative SDP_E* code otherwise,
 *     and never throws across the ABI; `sdp_last_error()` gives the text;
 *   - nothing is allocated, freed or retained by the library: all buffers are
 *     caller-owned and caller-sized;
 *   - no hidden synchronisation: work is enqueued on `stream`, the caller
 *     synchronises; entry points are thread-safe for distinct streams;
 *   - all arithmetic is IEEE fp64 with round-to-nearest and NO fused
 *     multiply-add contraction, in the reference's operation order
 *     (SURVEY.md App. A), so that cell indices / weights are bit-exact against
 *     the reference's compiled Cython routine.
 *
 * The reference has no FFI of its own: its only native seam is one Cython
 * function (stodynprog/dolointerpolation/multilinear_cython.pyx:17) and the
 * hot loop is Python (stodynprog/stodynprog.py:466-534, :639-691, :693-775).
 * Each entry point below cites the reference interface it replaces.
 */
#ifndef SDP_B200_H
#define SDP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SDP_ABI_VERSION 10
#define SDP_MAX_D 4 /* the reference dispatches d = 1..4 (multilinear_cython.pyx:36-47) */

/* error codes */
#define SDP_OK 0
#define SDP_EINVAL (-1)  /* bad argument (dimension, size, null pointer, alignment) */
#define SDP_ECUDA (-2)   /* a CUDA runtime call or kernel launch failed */
#define SDP_ENODEV (-3)  /* no CUDA device / wrong architecture */

/* Rectangular state grid: what MlinInterpolator stores (stodynprog.py:261-265):
 * smin = grid[0], smax = grid[-1], order = len(grid) per state variable.
 * Values on the grid are C-order (`J.ravel()`, stodynprog.py:272). */
typedef struct SdpGrid {
    int32_t d;                /* number of state variables, 1..SDP_MAX_D */
    int32_t order[SDP_MAX_D]; /* points per axis, each >= 2 */
    double smin[SDP_MAX_D];
    double smax[SDP_MAX_D];
} SdpGrid;

/* Per-state descriptor for the table build (host-built, device-read).
 * The user's dyn/cost return arrays broadcastable to (U1, ..., Unc, W) for one
 * state (or to (S, U1, ..., Unc, W) when the host evaluates a chunk of S states
 * in one call); they are uploaded un-broadcast into a staging buffer and
 * expanded on the device, which is what np.broadcast_arrays + astype(float) +
 * ravel do at stodynprog.py:281-283.  Slot k < d is next-state coordinate k,
 * slot d is the stage cost g.  Element (i_1..i_nc, w) of slot k of this state
 * is staging[src[k] + sum_c i_c*cs[k][c] + w*ws[k]]; the flat control index is
 * the C-order index over npts[0..nc) (stodynprog.py:686). */
#define SDP_MAX_C 4 /* control variables per system supported by the table build */
typedef struct SdpStateDesc {
    int64_t entry_off;                  /* layout A: first entry of the state's block */
    int64_t g_off;                      /* layout A: first entry of the state's g block */
    int64_t src[SDP_MAX_D + 1];         /* offset (in doubles) of each source array in staging */
    int32_t cs[SDP_MAX_D + 1][SDP_MAX_C]; /* source stride along control axis c (0 = broadcast) */
    int32_t ws[SDP_MAX_D + 1];          /* source stride along the perturbation index (0 = broadcast) */
    int32_t npts[SDP_MAX_C];            /* control grid dims of this state (1 for unused axes) */
    int32_t U;                          /* admissible control combinations = prod(npts) */
    int32_t Upad;                       /* layout A: U rounded up to a multiple of 4 */
} SdpStateDesc;

/* One unit of sweep work, processed by one warp.
 * Layout A: a run of controls of one state (`state` = local state index).
 * Layout B: a run of controls of one tile of 32 consecutive states
 *           (`state` = tile index, Upad unused).
 * Units with more controls than the chunk size are split into several items
 * whose partial (min, argmin) are combined by the finalize kernel. */
typedef struct SdpItem {
    int64_t entry_base; /* A: entry_off + u_begin;  B: tile_off + u_begin*W*32 */
    int64_t g_base;     /* A: g_off + u_begin;      B: tile_g_off + u_begin*32 (or = entry_base) */
    int32_t Upad;       /* A: row pitch of the state's block */
    int32_t u_begin;    /* first control of the run (A: multiple of 4) */
    int32_t u_count;    /* controls in the run */
    int32_t state;      /* A: local state index;  B: tile index */
} SdpItem;

#define SDP_LAYOUT_CONTROL_MINOR 0 /* "A": [state][w][u], lane <-> control   */
#define SDP_LAYOUT_STATE_MINOR 1   /* "B": [tile][u][w][32 states], lane <-> state */
/* Factored ("broadcast-compressed") variants, SURVEY.md §8(f)4: every next-state
 * coordinate depends either on (x,u) only or on (x,w) only and the stage cost
 * does not depend on w - true of every reference example (E_next = E + P_sto*dt,
 * P_next = a*P + w: examples/howto storage-AR1.ipynb:143; storage_control.py:49-65).
 * The dense (x,u,w) tables are then an outer sum of a (x,u) part and a (x,w)
 * part, which is what np.broadcast_arrays expands at stodynprog.py:281; the
 * factored layouts keep the two parts and the sweep kernel forms
 * cell = cell_u + cell_w and the weight vector on the fly.  Same arithmetic,
 * same order, bit-identical results; HBM traffic drops by about W. */
#define SDP_LAYOUT_CONTROL_MINOR_FACTORED 2 /* "AF": u-part [state][Upad], w-part [state][W] */
#define SDP_LAYOUT_STATE_MINOR_FACTORED 3   /* "BF": u-part [tile][u][32], w-part [tile][w][32] */
#define SDP_FACTORED_MAX_W_REG 9 /* BF keeps the w-part of a lane in registers: W <= 9 */
/* "CF", column-shared hoist: BF tables whose tiles run along state axis 0 - a tile holds
 * 32 consecutive rows of one COLUMN c (the flat C-order index over the state axes
 * 1..d-1) - for systems with u_mask == 1 whose (x,w) part does not depend on the axis-0
 * index (the storage examples: P_next = a*P + w does not involve E).  The inner
 * interpolation R(row, w) over the axes 1..d-1 is then the same for all the states of a
 * column: it is tabulated once per column and sweep (order[0] rows of W|1 doubles, held
 * in shared memory by the CTA that sweeps the column) and every backup of the column is
 * two shared-memory reads and one lerp instead of 2^d gathers and 2^d-1 lerps - the
 * operations of the reference's nested formula, evaluated once instead of once per
 * (state, control).  Bit-identical to the other layouts.
 * Tile order: the shard's rows are cut into one or more BANDS of consecutive rows; tiles
 * are ordered band by band, inside a band column by column, inside a column by rows
 * (band b, rows_b rows: tile = band_first_tile[b] + c*ceil(rows_b/32) + (row - first row)/32).
 * One band is the plain column-major order; several bands let a caller combine and copy
 * out the results of a band (a contiguous range of states) while later bands are swept. */
#define SDP_LAYOUT_COLUMN_FACTORED 4
/* doubles per column table: order[0] rows of (W|1) doubles + 9 of slack, rounded up to even */
#define SDP_COLUMN_PITCH(rows, W) ((((int64_t)(rows) * ((W) | 1)) + 9 + 1) & ~(int64_t)1)
#define SDP_COLUMN_PITCH2(rows, W) ((((int64_t)(rows) * ((W) | 1)) + ((rows) >> 1) + 10 + 1) & ~(int64_t)1) /* col_pairs */
#define SDP_COLUMN_MAX_SMEM_BYTES (200 * 1024) /* CF: 8 * SDP_COLUMN_PITCH[2](order[0], W) must fit */

/* Dense sweep tables of one shard of states (device pointers).
 *
 * Layout A (control-minor), per state block: entries [w][Upad], control fastest:
 *   cell[entry_off + w*Upad + u]                 int32 flat base-cell index
 *   lam [k*lam_plane + entry_off + w*Upad + u]   fp64 weight of state dim k
 *   g   [g_off + u]              if g_per_w == 0 (cost does not depend on w)
 *   g   [g_off + w*Upad + u]     if g_per_w == 1 (g_off == entry_off)
 *   Best when the gathers of neighbouring controls hit the same cell (many
 *   controls per state, fine control step): the 2^d corner loads of a warp
 *   are broadcasts.
 *
 * Layout B (state-minor), per tile of 32 consecutive states, U_t = max U:
 *   cell[tile_off + (u*W + w)*32 + lane]         lane = state - 32*tile
 *   lam [k*lam_plane + tile_off + (u*W + w)*32 + lane]
 *   g   [tile_g_off + u*32 + lane]  (g_per_w == 0)  or  g[tile_off + (u*W+w)*32 + lane]
 *   Best when neighbouring states land in neighbouring cells (many states, few
 *   controls): the corner loads of a warp are contiguous.
 *
 * Algorithmic bytes per admissible (x,u,w): 4 + 8*d + 8*(g_per_w ? 1 : 1/W).
 *
 * Factored layouts (g_per_w == 0; n_u = popcount(u_mask), n_w = d - n_u, both >= 1):
 *   u-part, entry e = entry_off + u (AF, per state, Upad entries)
 *                   = tile_off + u*32 + lane (BF, per tile, U_t*32 entries):
 *     cell [e]                    sum over u-type coordinates k of q_k*M_k
 *     lam  [j*lam_plane + e]      weight of the j-th u-type coordinate (increasing k)
 *     g    [e]                    stage cost
 *   w-part, entry f = state*W + w (AF) = (tile*W + w)*32 + lane (BF):
 *     cell_w[f], lam_w[j*lam_w_plane + f]   same for the w-type coordinates
 *   Items: entry_base = g_base = first u-part entry of the run.
 *   Actual bytes per (x,u,w): (12 + 8*n_u)/W + (4 + 8*n_w)/U(x).
 *
 * Layout CF: see SDP_LAYOUT_COLUMN_FACTORED and the last fields below. */
typedef struct SdpTables {
    const int32_t* cell;
    const double* lam;
    int64_t lam_plane;
    const double* g;
    int32_t g_per_w;
    int32_t W;           /* perturbation nodes (1 for a deterministic system) */
    int32_t expect;      /* 1: J = sum_w p_w*(g+J'); 0: deterministic, J = g+J' */
    int32_t layout;      /* SDP_LAYOUT_* */
    const double* p;     /* [W] probabilities (ignored when expect == 0) */
    const SdpItem* items;
    int64_t n_items;
    const int64_t* item_begin; /* A: [n_states+1], B: [n_tiles+1]: items of unit i are item_begin[i]..item_begin[i+1]-1 */
    int64_t n_states;    /* states in this shard */
    const int32_t* U;    /* [n_states] admissible controls per state (layout B masking) */
    /* factored layouts only */
    int32_t u_mask;        /* bit k set: coordinate k depends on (x,u) only; clear: on (x,w) only */
    int32_t col_pairs;     /* layout CF: 1 = two rows per lane (see pos_row below), 0 = one */
    const int32_t* cell_w;
    const double* lam_w;
    int64_t lam_w_plane;
    /* HOST copy of p[W] (the same values as `p`).  Required by layout BF, whose
     * kernel takes the probabilities as launch constants; ignored otherwise. */
    const double* p_host;
    /* Layout CF only.  The shard is `n_states / n_cols` whole rows of axis 0 (local
     * state i = row*n_cols + column, as in the C-order grid); units/items/u-part/w-part
     * are those of layout BF over the tiles described above, `U` is indexed by POSITION
     * tile*32 + lane (0 on the padding lanes of a column's last tile in a band); item.Upad
     * holds the COLUMN of the item's tile.  The w-part read for column c is that of lane 0
     * of tile c*tiles_per_col, its first tile in the first band (the caller checks that
     * the whole column agrees).
     * Streaming pass (sdp_sweep_partials): one CTA sweeps the items
     * seg_begin[b] .. seg_begin[b+1]-1 (absolute indices into `items`; items are ordered by
     * tile) and loads its column table whenever the column changes: run_end[i] is the end
     * of the run of items sharing the band and column of item i.
     * Combine pass (sdp_sweep_finalize[_p2p]): called ONCE PER BAND with a view of the
     * band - item_begin advanced to the band's first tile, n_states / tiles_per_col those
     * of the band, outputs advanced to the band's first state. */
    int32_t n_cols;
    int32_t tiles_per_col;     /* streaming pass: of the first band; combine pass: of the band */
    const int64_t* seg_begin;  /* [n_segs + 1] */
    int64_t n_segs;
    /* scratch, written by every sweep: the inner-interpolation tables of all columns,
     * [n_cols][SDP_COLUMN_PITCH(order[0], W)] doubles (caller-owned, 16-byte aligned).  A
     * coalesced pre-pass (sdp_column_table, lanes along the columns, where the gathers of
     * neighbouring columns are contiguous) fills it from J_prev and each CTA copies the
     * table of its current column into shared memory. */
    double* col_table;
    const int64_t* run_end;    /* [n_items] */
    int32_t col_table_ready;   /* streaming pass: 0 = run the pre-pass first, 1 = col_table is current */
    /* streaming pass, optional launch shape: low 16 bits = threads per CTA (0: library default),
     * bit 16 = hand the items of a run out round-robin instead of first come first served */
    int32_t col_launch_hint;
    /* streaming pass, optional [n_items]: the ORDER in which the item list is walked - seg_begin and
     * run_end then refer to positions p of this order, position p being item item_order[p], and a
     * run is a stretch of positions whose items share a column (any bands).  NULL: positions are
     * item indices.  Lets a device-resident sweep visit the bands of a column back to back (one
     * table load per column) while the tables stay ordered band by band for the combine. */
    const int64_t* item_order;
    /* Layout CF with col_pairs = 1 ("two rows per lane").  A lane of the streaming pass then owns
     * the positions 2j, 2j+1 of a tile: two rows of the column that are neighbours on axis 0, so
     * that the table rows their backups read overlap - R[q], R[q+1] and R[q'], R[q'+1] with
     * q' in {q, q+1} - and 3 shared-memory reads serve 2 backups (anything else is handled, with
     * a 4th read).  Positions are no longer rows: the caller pairs rows as it sees fit (rows
     * with the same control grid size) and pads, `pos_row[p]` = row of the band held by position
     * p of EVERY column, -1 on padding; tiles per column is even, the two tiles of a pair are
     * cut into the same runs of controls, and the streaming pass walks `item_order` (required),
     * which lists the items of the FIRST tile of every pair only: item.g_base of such an item is
     * the index of the same run in the second tile.  The column tables are swizzled: row q at
     * q*(W|1) + (q >> 1), SDP_COLUMN_PITCH2 doubles per column.
     * Combine pass: pos_row advanced to the band's first position. */
    const int32_t* pos_row;
    /* Layout CF, optional scratch written with col_table (caller-owned, 16-byte aligned, NULL: no
     * pruning): [n_cols][order[0]] pairs of doubles, for table row q of a column
     *   m(q) = sum_w p_w * min(R[q][w], R[q+1][w])      (w in order, rounded as written)
     *   A(q) = max_w max(|R[q][w]|, |R[q+1][w]|)        (NaN when one of them is NaN)
     * and (0, NaN) for the last row.  m(q) + g*sum(p) bounds from below the value of every
     * control whose axis-0 weight is in [0, 1] and that interpolates between rows q and q+1:
     * the streaming pass skips a control when that bound, less a rounding margin, is already
     * worse than the best value of the lane (DESIGN.md section 4; option "col_prune").  Used
     * only with one row per lane, expect == 1 or W == 1, p_w in [0, 1], and when table and
     * bound together fit SDP_COLUMN_MAX_SMEM_BYTES; ignored otherwise. */
    double* col_bound;
} SdpTables;

/* ABI / build identification. */
int sdp_version(void);
const char* sdp_last_error(void);
/* Number of kernels launched by this library since load (for bench accounting). */
int64_t sdp_launch_count(void);
/* Name (template arguments, CTA shape) of the streaming kernel that the calling thread's last
 * sdp_sweep / sdp_sweep_partials launched: what a bench line or a profile summary must call
 * it.  Valid until that thread's next launch. */
const char* sdp_last_kernel(void);

/* Launch tuning (developer knob; defaults are read from SDP_* environment
 * variables): "upl" (2|4), "wb" (1|2|3|5), "tma" (layout-B kernel: 0 straight
 * LDG, 1 TMA-fed ring, 2 software-pipelined LDG = default), "rb" (2|4|8),
 * "tma_rows" (4|8), "tma_stages" (2..16), "tma_warps" (1..16), "hoist" (layout AF
 * with u_mask == 1: per-item table of inner interpolations, 0|1), "hoist_upl" (2|4),
 * "hoist_const" (0|1: constant-W variant of that kernel for W <= 9),
 * "col_threads" (layout CF: threads per CTA, 128..768; 0 = default, 768, or 640 when pruning), "col_ub" (controls per iteration, 1|2),
 * "col_pf" (groups of col_ub controls in flight, 1|2), "col_dynamic" (0|1: the warps of a CTA
 * take the items of a column round-robin / first come first served), "col_prepass" (column tables
 * from the coalesced pre-pass, copied into shared memory by the TMA engine = 2, default, or by
 * vector loads = 1; 0: every CTA gathers its own from J_prev),
 * "col_prune" (layout CF with col_bound: skip the controls that provably lose, 1 = default, or
 * evaluate every control, 0; the results are the same),
 * "col_prune_stats" (0|1: count the warp steps of the pruning sweep and those skipped, read and
 * reset by sdp_col_prune_counts; off by default, for measurements only),
 * "p2p_timeout_s" (bound of the peer-flag waits, default 600 s, then the kernel traps),
 * "chain_threads" (sdp_chain_sample: threads per CTA, 32..1024 in multiples of 32; 0 = default,
 * 256; the results do not depend on it).
 * Not thread-safe against concurrent launches. */
int sdp_set_option(const char* name, int value);
/* With "col_prune_stats" on: the warp steps (groups of col_ub controls of one item) that the
 * pruning column sweeps have met, and how many of them skipped the evaluation, since the previous
 * call.  Synchronizes the device.  Both are 0 when nothing was counted. */
int sdp_col_prune_counts(int64_t* steps, int64_t* skipped);

/* K0a - cell search on explicit points.
 * Replaces the cell-search half of multilinear_interpolation_{1..4}d
 * (multilinear_cython.pyx:72-79, :117-131, :177-193, :257-278).
 * s: device [d][n]; cell: device [n]; lam: device [d][n]. */
int sdp_cell_setup(const SdpGrid* grid, int64_t n, const double* s, int32_t* cell,
                   double* lam, void* stream);

/* K0b - table build for a chunk of states: broadcast-expand the staged
 * dyn/cost outputs (stodynprog.py:674-677 + :281-283) and run the cell search.
 * desc: device [n_states]; staging: device doubles; outputs as in SdpTables.
 * Padding entries get cell 0, lam 0, g 0.
 * Layout A: */
int sdp_build_tables(const SdpGrid* grid, int32_t W, int32_t g_per_w, int64_t n_states,
                     const SdpStateDesc* desc, const double* staging, int32_t* cell,
                     double* lam, int64_t lam_plane, double* g, int32_t max_Upad,
                     void* stream);
/* Layout B: `n_tiles` tiles of 32 states; desc[i] describes state i of the
 * chunk (n_states <= 32*n_tiles, the last tile may be partial); tile arrays are
 * device [n_tiles]: first entry, first g entry, U_t = max U of the tile. */
int sdp_build_tables_tiled(const SdpGrid* grid, int32_t W, int32_t g_per_w, int64_t n_states,
                           const SdpStateDesc* desc, const double* staging, int64_t n_tiles,
                           const int64_t* tile_off, const int64_t* tile_g_off,
                           const int32_t* tile_U, int32_t max_tile_U, int32_t* cell,
                           double* lam, int64_t lam_plane, double* g, void* stream);

/* Factored layouts: the same expansion, kept as a (x,u) part and a (x,w) part.
 * Coordinate k of entry (u) is read at w index 0 when bit k of u_mask is set,
 * coordinate k of entry (w) at flat control index 0 otherwise; g at w index 0.
 * The caller guarantees (and checks on the descriptors) that the staged arrays
 * do not depend on the other index.  cell_w / lam_w point at the w-part of the
 * chunk's first state (AF) or first tile (BF).
 * AF: desc[i].entry_off = first u-part entry of state i, Upad entries. */
int sdp_build_tables_factored(const SdpGrid* grid, int32_t W, int32_t u_mask, int64_t n_states,
                              const SdpStateDesc* desc, const double* staging, int32_t* cell,
                              double* lam, int64_t lam_plane, double* g, int32_t max_Upad,
                              int32_t* cell_w, double* lam_w, int64_t lam_w_plane, void* stream);
/* BF: tile_off[t] = first u-part entry of tile t of the chunk, tile_U[t] = max U. */
int sdp_build_tables_factored_tiled(const SdpGrid* grid, int32_t W, int32_t u_mask, int64_t n_states,
                                    const SdpStateDesc* desc, const double* staging, int64_t n_tiles,
                                    const int64_t* tile_off, const int32_t* tile_U,
                                    int32_t max_tile_U, int32_t* cell, double* lam,
                                    int64_t lam_plane, double* g, int32_t* cell_w, double* lam_w,
                                    int64_t lam_w_plane, void* stream);

/* K1 - one Bellman sweep over a shard of states.
 * Replaces the state loop of DPSolver.value_iteration (stodynprog.py:511-515)
 * with _value_at_state_vect (:639-691): gather + nested lerp of J_prev
 * (pyx:81-88, :133-140, :195-208, :280-300), + g, expectation over w
 * (np.inner, :682), first-minimum argmin over the control product (:686).
 * J_prev: device [prod(order)], the full previous value function.
 * part_val/part_idx: device scratch [n_items] (layout A) or [32*n_items] (layout B).
 * J_out: device [n_states]; argmin_out: device [n_states] flat C-order index
 * into the state's control product.  (Layout CF: single-band tables only.) */
int sdp_sweep(const SdpGrid* grid, const SdpTables* tab, const double* J_prev,
              double* part_val, int32_t* part_idx, double* J_out, int32_t* argmin_out,
              void* stream);
/* Layout CF: the pre-pass of the streaming pass alone (fills tab->col_table from J_prev),
 * for callers that sweep the item list in several launches with col_table_ready = 1.
 * Part of K1: it evaluates, once per grid column and perturbation node, the inner levels of
 * the nested lerp of multilinear_interpolation_{2,3}d (multilinear_cython.pyx:133-140,
 * :195-208) that `J_next_interp(*x_next)` (stodynprog.py:677) repeats for every control. */
int sdp_column_table(const SdpGrid* grid, const SdpTables* tab, const double* J_prev, void* stream);
/* The two launches of sdp_sweep, separately (so that a caller can bracket the
 * streaming kernel alone with events): per-item partial minima, then the
 * per-state combine. */
int sdp_sweep_partials(const SdpGrid* grid, const SdpTables* tab, const double* J_prev,
                       double* part_val, int32_t* part_idx, void* stream);
int sdp_sweep_finalize(const SdpTables* tab, const double* part_val, const int32_t* part_idx,
                       double* J_out, int32_t* argmin_out, void* stream);

/* Multi-GPU exchange over peer memory (NVLink 5 / NVSwitch), SURVEY.md §8e.
 * The state grid is cut into one slab per rank; every rank keeps the whole J.
 * Instead of an NCCL all-gather after the sweep, the per-state combine kernel
 * stores each new J value straight into the J buffer of EVERY rank (peer-mapped
 * pointers of a symmetric allocation), and the last CTA to finish publishes the
 * rank's epoch in every rank's flag array; consumers wait on their local flags.
 * All pointers are device pointers valid on the calling rank's GPU. */
#define SDP_MAX_PEERS 8
typedef struct SdpPeers {
    int32_t world, rank;
    double* J[SDP_MAX_PEERS];         /* [n_grid] destination buffer on every rank (J[rank] = local) */
    uint64_t* flags[SDP_MAX_PEERS];   /* [world] flag array on every rank; this rank writes entry `rank` */
    uint64_t* epoch;                  /* local: exchanges/barriers completed by this rank */
    uint32_t* done;                   /* local: CTA completion counter, zero between launches */
    /* optional (all NULL: off): [n_grid] int32 argmin buffer on every rank.  The fused combine then
     * stores each state's argmin next to its J on every rank, so that every rank holds the whole
     * policy and the host results can be mapped and copied out by all ranks in parallel. */
    int32_t* A[SDP_MAX_PEERS];
} SdpPeers;
/* Fused per-state combine + all-gather: as sdp_sweep_finalize, but J goes to
 * peers->J[r][state_begin + i] for every rank r; then epoch += 1 and the new
 * epoch is released (system scope) into flags[r][rank] for every r.
 * Every rank must issue the same sequence of finalize_p2p / barrier calls. */
int sdp_sweep_finalize_p2p(const SdpTables* tab, const double* part_val, const int32_t* part_idx,
                           int32_t* argmin_out, const SdpPeers* peers, int64_t state_begin,
                           void* stream);
/* The same for a shard made of whole COLUMNS of the grid (layout CF, one band, n_cols local
 * columns): local state i = row*n_cols + lc is grid state row*glob_cols + col_begin + lc, and
 * that is where its J goes in every rank's buffer.  (Sharding by columns keeps the cost of the
 * column tables - pre-pass and loads - proportional to the shard.) */
int sdp_sweep_finalize_p2p_cols(const SdpTables* tab, const double* part_val, const int32_t* part_idx,
                                int32_t* argmin_out, const SdpPeers* peers, int64_t glob_cols,
                                int64_t col_begin, void* stream);
/* Stream-ordered wait until every rank has published the local epoch (i.e. until
 * the slabs written by the last sdp_sweep_finalize_p2p of all ranks have landed). */
int sdp_p2p_wait(const SdpPeers* peers, void* stream);
/* sdp_p2p_wait(wait_for) followed by sdp_sweep_partials(...), with the wait folded into the first
 * kernel that reads J_prev where the layout has one that can carry it (layout CF: every CTA of
 * the column-table pre-pass starts with the flag wait) - one launch less per sweep of a
 * device-resident iteration.  Same results as the two calls. */
int sdp_sweep_partials_after(const SdpGrid* grid, const SdpTables* tab, const double* J_prev,
                             double* part_val, int32_t* part_idx, const SdpPeers* wait_for,
                             void* stream);
/* Hand a piece of J to the peers: src[offset .. offset+n) (this rank's device copy) is stored at the
 * same indices of every OTHER rank's peers->J buffer, then the epoch is published as by
 * sdp_sweep_finalize_p2p (follow with sdp_p2p_wait; every rank calls it, n may be 0).  Used when
 * every rank uploads 1/N of the next sweep's input from host memory shared by the ranks. */
int sdp_p2p_broadcast(const double* src, int64_t offset, int64_t n, const SdpPeers* peers, void* stream);
/* Stream-ordered barrier over the ranks: epoch += 1, publish, wait. */
int sdp_p2p_barrier(const SdpPeers* peers, void* stream);

/* K1' - fixed-policy backups (policy evaluation), `n_iter` iterations.
 * Replaces the body of DPSolver.eval_policy (stodynprog.py:743-763).
 * Tables are [w][n_states] planes (state index fastest):
 *   cell[w*n_states + i], lam[k*lam_plane + w*n_states + i],
 *   g[i] (g_per_w == 0) or g[w*n_states + i].
 * J_a / J_b: device [n_grid] ping-pong buffers; iteration k reads one and writes
 * states [state_begin, state_begin + n_states) of the other; on return the
 * result is in J_a if n_iter is even, J_b if odd.
 * rel_dp != 0: after each iteration J_ref_hist[k] = J[ref_index]; J -= that
 * (stodynprog.py:760-762), fused into the backup kernel (every block recomputes the
 * reference state's backup, same operations, same bits); requires the shard to be the
 * whole grid.
 * J_ref_hist: device [n_iter] (may be NULL when rel_dp == 0). */
int sdp_policy_eval(const SdpGrid* grid, int32_t W, int32_t g_per_w, const double* p,
                    const int32_t* cell, const double* lam, int64_t lam_plane,
                    const double* g, int64_t n_states, int64_t state_begin, int64_t n_grid,
                    double* J_a, double* J_b, int32_t n_iter, int32_t rel_dp,
                    int64_t ref_index, double* J_ref_hist, void* stream);

/* One fixed-policy backup of this rank's slab fused with the all-gather over peer
 * memory: as one iteration of sdp_policy_eval, but the new values go to
 * peers->J[r][state_begin + i] for every rank r and the rank's epoch is published
 * (same protocol as sdp_sweep_finalize_p2p; follow with sdp_p2p_wait).
 * J_in: device [n_grid], the full previous value function on this rank.
 * Relative DP (ref_cell != NULL): every rank passes its own copy of the table entries
 * of the reference state - ref_cell [W], ref_lam [d][W], ref_g [W] (g_per_w) or [1] -
 * and the kernel subtracts that state's new value from everything it stores
 * (stodynprog.py:760-762); J_ref_out[0] receives it. */
int sdp_policy_eval_p2p(const SdpGrid* grid, int32_t W, int32_t g_per_w, const double* p,
                        const int32_t* cell, const double* lam, int64_t lam_plane,
                        const double* g, int64_t n_states, int64_t state_begin, int64_t n_grid,
                        const double* J_in, const SdpPeers* peers, const int32_t* ref_cell,
                        const double* ref_lam, const double* ref_g, double* J_ref_out,
                        void* stream);

/* K1'' - forward (adjoint) application of a fixed policy: propagation of a state distribution.
 * New feature, no reference counterpart: the reference estimates what a policy does to the
 * system by simulating one trajectory point at a time (examples/20 .../storage_control.py:217,246).
 * The fixed-policy backup of sdp_policy_eval is J <- g_bar + P J with the interpolated Markov
 * chain P of the policy tables (same [w][n] planes: cell, lam, g, p); these entry points apply
 * the transpose, mu <- P^T mu:
 *   (P^T mu)(y) = sum over (x, w, eps in {0,1}^d) with cell[w*n + x] + sum_k eps_k*M_k = y of
 *                 mu(x) * coef(x, w, eps)
 *   coef(x, w, eps) = p_w * f_0 * f_1 * ... * f_{d-1}, multiplied left to right,
 *                     f_k = eps_k ? lam_k : (1 - lam_k),  lam_k = lam[k*lam_plane + w*n + x]
 * (bit k of eps is the corner along axis k, M_k the C-order strides).  Weights are not clamped:
 * outside the grid box the coefficients extrapolate and may be negative, exactly as the backup.
 * The operator is stored as CSR by DESTINATION y, every (x, w, eps) kept (nnz = n*W*2^d, known up
 * front; n*W*2^d < 2^31), entries of a row ordered by the source key (x*W + w)*2^d + eps, so the
 * build is deterministic.  Rows longer than SDP_FWD_PIECE entries (extrapolated next states all
 * land in the first or last cell) are cut into pieces of SDP_FWD_PIECE entries, summed
 * separately and combined in piece order: every sum has a fixed association, independent of the
 * launch shape, and there are no floating-point atomics - results are bit-identical run to run.
 * All buffers are caller-owned device memory (the struct itself is a host pointer). */
#define SDP_FWD_PIECE 1024
typedef struct SdpForwardOp {
    int64_t n;              /* states (the whole grid: one rank) */
    int64_t nnz;            /* n * W * 2^d */
    int64_t* row_ptr;       /* [n+1] entries of row y: row_ptr[y] .. row_ptr[y+1]-1 */
    int32_t* src;           /* [nnz] source state x of each entry */
    double* coef;           /* [nnz] coefficient of each entry */
    double* gbar;           /* [n] expected stage cost g_bar(x) = sum_w p_w*g(x,w), summed in w order */
    int64_t* piece_first;   /* [n+1] pieces of row y: piece_first[y] .. piece_first[y+1]-1 (none for short rows) */
    int32_t* piece_row;     /* [max_pieces] row of each piece */
    int64_t max_pieces;     /* from sdp_forward_sizes */
    int64_t n_pieces;       /* piece_first[n]: read back by the caller after the build, used by the steps */
} SdpForwardOp;

/* Sizes of the buffers of a forward operator on a grid of n states, W nodes, d axes: nnz,
 * max_pieces, the bytes of build scratch and the doubles of step scratch.  Needs the device
 * current (the scratch of the library's sort is sized for it). */
int sdp_forward_sizes(int32_t d, int32_t W, int64_t n, int64_t* nnz, int64_t* max_pieces,
                      int64_t* build_scratch_bytes, int64_t* step_scratch_doubles);
/* Build op (row_ptr, src, coef, gbar, piece_first, piece_row) from the policy tables of the
 * whole grid, in the layout sdp_policy_eval takes (g_per_w as there).  Count per destination
 * (integer atomics), exclusive scan, fill through per-row cursors, sort of every row by source
 * key, coefficients; then the piece index of the long rows.  scratch: device, scratch_bytes >=
 * build_scratch_bytes, 256-byte aligned; nothing of it is needed afterwards. */
int sdp_forward_build(const SdpGrid* grid, int32_t W, int32_t g_per_w, const double* p,
                      const int32_t* cell, const double* lam, int64_t lam_plane, const double* g,
                      const SdpForwardOp* op, void* scratch, int64_t scratch_bytes, void* stream);
/* n_steps applications of P^T, ping-pong between mu_a (holds mu_0) and mu_b: step k reads mu_k
 * and writes mu_{k+1}; on return mu_n is in mu_a if n_steps is even, mu_b if odd.
 * cost_out: device [n_steps], cost_out[k] = <mu_k, g_bar> (expected stage cost of step k);
 * resid_out: device [1] or NULL, sum_y |mu_n(y) - mu_{n-1}(y)| of the last step;
 * hist: device [(n_steps+1)*n] or NULL, hist[k*n + y] = mu_k(y);
 * scratch: device [step_scratch_doubles].  Launches per step: a piece pass (when n_pieces > 0),
 * the row pass (a team of 8 lanes per row, 256 rows per CTA, per-CTA partial sums of the cost
 * and the residual), a one-CTA reduction of those partials. */
int sdp_forward_steps(const SdpForwardOp* op, double* mu_a, double* mu_b, int32_t n_steps,
                      double* cost_out, double* resid_out, double* hist, double* scratch, void* stream);

/* K1''' - sample paths of the chain of a fixed policy (Monte-Carlo trajectories).
 * New feature, no reference counterpart as a kernel: the reference simulates the policy on the host
 * (examples/20 .../storage_control.py:217,246).  The chain is the one of sdp_forward_*, sampled:
 * from state x, draw node w with probability p_w (u in [0,1), t = u*cdf[W-1], w the first index
 * with t < cdf[w], W-1 if none), then for every axis k draw v_k in [0,1) and take the upper corner
 * when v_k < clamp(lam_k, 0, 1); the next state is cell + sum_k eps_k*M_k and the path's total
 * gets acc = acc + g(x, w).  A transition with some lam_k outside [0,1] (an extrapolated next
 * state, projected onto the grid box by the clamp) is counted as clamped; a NaN lam_k gives
 * eps_k = 0 and counts the transition as NaN.
 * Random numbers: Philox-4x32-10, key = seed (low word first), counter (path, step, call, 0),
 * step the global step, call = 0, 1, 2 the calls of the step: 1 + d doubles, double j from words
 * 2(j%2), 2(j%2)+1 of call j/2 as ((lo | hi << 32) >> 11) * 2^-53.  Initial states drawn from a
 * CDF use step SDP_CHAIN_INIT_STEP.  A path's results depend only on (seed, path index, tables),
 * not on the launch shape; the only atomics are integer counter sums. */
#define SDP_CHAIN_INIT_STEP 0xFFFFFFFFu
/* doubles per (x, w) record: [cell (int32 in the low word) | lam_0 .. lam_{d-1} | g | pad to even]:
 * 32 bytes (one sector) for d <= 2, 48 for d = 3, 4 */
#define SDP_CHAIN_REC(d) (2 * (((d) + 3) / 2))
/* Pack the [w][n] policy-table planes (layout of sdp_policy_eval, g_per_w as there) into one record
 * per (x, w), record e = w*n + x at rec + e*SDP_CHAIN_REC(d).  rec: device, 16-byte aligned,
 * n*W*SDP_CHAIN_REC(d) doubles, owned by the caller. */
int sdp_chain_pack(const SdpGrid* grid, int32_t W, int32_t g_per_w, const int32_t* cell, const double* lam,
                   int64_t lam_plane, const double* g, int64_t n, double* rec, void* stream);
/* Advance M paths by n_steps steps, global steps step0 .. step0 + n_steps - 1, one thread per path,
 * the state in registers.  cdf: device [W], cumulative node probabilities (host np.cumsum).
 * fresh != 0: paths start at global step step0 with total 0 and hit -1, from state[i] or, when
 * start_cdf (device [n], cumulative, in C order) is given, from a state drawn with it (written to
 * state[i]); fresh == 0: resume from state, total, hit as a previous launch left them.
 * At every global step s in [step0, step0 + n_steps], before the transition out of s:
 *   target (device bit mask, bit y%32 of word y/32, or NULL): hit[i] = s if hit[i] < 0 and the
 *   state is in the target;  rec_steps (device [n_rec], strictly increasing, or NULL): when
 *   s == rec_steps[j], rec_out[j*M + i] = the state.
 * On return state / total / hit hold the state at step0 + n_steps, the summed stage costs and the
 * first step in the target.  counters (device [2], accumulated, zeroed by the caller):
 * counters[0] += clamped transitions, counters[1] += NaN transitions.  1 <= M < 2^31, n_steps >= 0,
 * step0 + n_steps < 2^32 - 1. */
int sdp_chain_sample(const SdpGrid* grid, int32_t W, const double* cdf, const double* rec, int64_t M,
                     int32_t n_steps, int64_t step0, uint64_t seed, int32_t fresh, const double* start_cdf,
                     const uint32_t* target, const int32_t* rec_steps, int32_t n_rec, int32_t* state,
                     double* total, int32_t* hit, int32_t* rec_out, unsigned long long* counters,
                     void* stream);

/* K3 - argmin index -> control values, the `u_grids[i].flatten()[ind_opt[i]]` of
 * stodynprog.py:686-689 for every state at once.  lo/hi: device [n][nc] box
 * bounds, npts: device [n][nc] grid sizes (what control_grids computed,
 * stodynprog.py:445-460), argmin: device [n] flat C-order index.
 * pol: device [n][nc], bit-identical to np.linspace(lo, hi, npts)[idx]
 * (or the centre point (lo+hi)/2 when npts == 1). */
int sdp_policy_values(int64_t n, int32_t nc, const double* lo, const double* hi,
                      const int32_t* npts, const int32_t* argmin, double* pol, void* stream);

/* One rank, layout CF, results handed out by COLUMN pieces (the host path of value_iteration:
 * a piece is swept, combined and on its way to the host while the next pieces compute).  `tab` is a
 * view of the tables on the columns [col_begin, col_begin + tab->n_cols) of a grid of glob_cols
 * columns: item_begin starts at the first tile of col_begin, one band of rows.  The per-state
 * combine of sdp_sweep_finalize for those columns; J_out / argmin_out are WHOLE-GRID arrays in
 * grid order (state row*glob_cols + col).  nc > 0: the argmin is also mapped to control values
 * as by sdp_policy_values (lo / hi / npts / pol: whole-grid [state][nc]) - the
 * `u_grids[i].flatten()[ind_opt[i]]` of stodynprog.py:686-689 fused into the combine.
 * beside_sweep != 0: a later piece is being swept on another stream meanwhile; the launch then uses
 * CTAs of 128 threads x 32 registers, which fit next to a resident CTA of the streaming kernel (one
 * per SM, 768 threads x 80 registers), so the combine does not wait for an SM to drain. */
int sdp_sweep_finalize_cols(const SdpTables* tab, const double* part_val, const int32_t* part_idx,
                            double* J_out, int32_t* argmin_out, int64_t glob_cols, int64_t col_begin,
                            int32_t nc, const double* lo, const double* hi, const int32_t* npts,
                            double* pol, int32_t beside_sweep, void* stream);

/* `height` rows of `width` bytes from src (row pitch spitch bytes) to dst (row pitch dpitch),
 * asynchronously on the stream; either side device or page-locked host memory.  Puts a column
 * piece of a result where it belongs in the caller's C-order host array (the reference returns
 * J_k and pol_k as C-order arrays over the state grid, stodynprog.py:496-499). */
int sdp_memcpy_2d(void* dst, int64_t dpitch, const void* src, int64_t spitch, int64_t width,
                  int64_t height, void* stream);

/* Relative-DP normalisation: ref_out[0] = J[ref_index]; J[i] -= ref_out[0]
 * (stodynprog.py:523-525, :760-762).  J: device [n]. */
int sdp_rel_shift(double* J, int64_t n, int64_t ref_index, double* ref_out, void* stream);

/* Sup-norm of the update, max_i |a[i] - b[i]| (NaN differences ignored), written
 * to out[0].  New feature (the reference never computes a residual). */
int sdp_supnorm_diff(const double* a, const double* b, int64_t n, double* out, void* stream);

/* K2 - multilinear interpolation of n_v value rows at n_s points.
 * Replaces multilinear_interpolation (multilinear_cython.pyx:17-49).
 * values: device [n_v][prod(order)]; s: device [d][n_s]; out: device [n_v][n_s]. */
int sdp_interp(const SdpGrid* grid, int64_t n_v, const double* values, int64_t n_s,
               const double* s, double* out, void* stream);
/* fp32 specialisation of the same routine (the `float` branch of the fused
 * type `floating`, multilinear_cython.pyx:12-14,22-25). smin/smax are rounded
 * to fp32 as the reference's float memoryviews would hold them. */
int sdp_interp_f32(const SdpGrid* grid, int64_t n_v, const float* values, int64_t n_s,
                   const float* s, float* out, void* stream);

/* K2 for a handful of points, on the HOST: values, s and out are host pointers, nothing touches
 * the GPU.  Same operations in the same order as sdp_interp / sdp_interp_f32 (bit-identical
 * results).  For the one-point-at-a-time calls of the reference's simulation loops
 * (examples/20 Searev storage control/storage_control.py:217,246 evaluate
 * `interp_on_state(pol)(x)` per time step), where a launch plus two PCIe crossings per point
 * would make the drop-in slower than multilinear_cython.pyx:17-49 itself.  Not a fallback: the
 * Python front-end uses it below a point-count threshold only, and the library is still required. */
int sdp_interp_host(const SdpGrid* grid, int64_t n_v, const double* values, int64_t n_s,
                    const double* s, double* out);
int sdp_interp_host_f32(const SdpGrid* grid, int64_t n_v, const float* values, int64_t n_s,
                        const float* s, float* out);

#ifdef __cplusplus
}
#endif
#endif /* SDP_B200_H */
