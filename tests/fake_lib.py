"""numpy model of the C ABI (include/sdp_b200.h) for host-logic tests.

TEST INFRASTRUCTURE ONLY.  It lets the tests drive the product's *host* code
(tabulation, descriptors, work items, slabs, collectives, argmin -> control
values) on a machine without a GPU, by standing in for libsdp_b200.so behind
`Engine(_test_lib=...)`.  It reads and writes the caller's (CPU torch) buffers
through raw pointers with exactly the table layout the header documents, and
does its arithmetic with the C oracle.  It is deliberately slow and simple.
"""
import ctypes

import numpy as np

from oracle import oracle as oc
from stodynprog_b200 import _cabi


def _arr(ptr, n, ctype):
    p = ptr.value if hasattr(ptr, "value") else ptr
    if n == 0 or not p:
        return np.zeros(0, dtype=ctype)
    return np.ctypeslib.as_array((ctype * n).from_address(p))


def _grid(gref):
    g = gref._obj
    d = g.d
    return d, np.array(g.smin[:d]), np.array(g.smax[:d]), np.array(g.order[:d], dtype=np.int64)


def _better(av, ai, bv, bi):
    an, bn = av != av, bv != bv
    if an or bn:
        return (ai < bi) if (an and bn) else an
    if av < bv:
        return True
    if av > bv:
        return False
    return ai < bi


class FakeLib(object):
    def __init__(self):
        self.launches = 0
        self.err = b""

    def sdp_version(self):
        return _cabi.SDP_ABI_VERSION

    def sdp_last_error(self):
        return self.err

    def sdp_launch_count(self):
        return self.launches

    def sdp_last_kernel(self):
        return b"fake_lib (numpy model of the ABI)"

    def sdp_cell_setup(self, gref, n, s, cell, lam, stream):
        d, smin, smax, orders = _grid(gref)
        S = _arr(s, d * n, ctypes.c_double).reshape(d, n)
        c, l = oc.cell_search(smin, smax, orders, S)
        _arr(cell, n, ctypes.c_int32)[:] = c
        _arr(lam, d * n, ctypes.c_double)[:] = l.reshape(-1)
        self.launches += 1
        return 0

    @staticmethod
    def _src_index(r, k, U, W, nc_max=_cabi.SDP_MAX_C):
        """(W, U) array of staging offsets of slot k for state record r"""
        u = np.arange(U)
        off = np.zeros(U, dtype=np.int64) + int(r["src"][k])
        rem = u.copy()
        for c in range(nc_max - 1, -1, -1):
            n = int(r["npts"][c])
            off += (rem % n) * int(r["cs"][k][c])
            rem //= n
        return off[None, :] + np.arange(W)[:, None] * int(r["ws"][k])

    def _expand_state(self, r, d, W, stag, smin, smax, orders):
        U = int(r["U"])
        assert U == int(np.prod(r["npts"]))
        coords = np.stack([stag[self._src_index(r, k, U, W)].reshape(-1) for k in range(d)])
        c, l = oc.cell_search(smin, smax, orders, coords)
        gsrc = stag[self._src_index(r, d, U, W)]
        return c.reshape(W, U), l.reshape(d, W, U), gsrc

    def _staging(self, D, d, W, staging):
        top = 0
        for r in D:
            U = max(int(r["U"]), 1)       # U = 0: a padding position of layout CF (only its w-part is read)
            for k in range(d + 1):
                top = max(top, int(self._src_index(r, k, U, W).max()) + 1)
        return _arr(staging, top, ctypes.c_double)

    def sdp_build_tables(self, gref, W, g_per_w, n_states, desc, staging, cell, lam, lam_plane, g,
                         max_Upad, stream):
        d, smin, smax, orders = _grid(gref)
        D = np.frombuffer((ctypes.c_uint8 * (n_states * _cabi.STATE_DESC_DTYPE.itemsize))
                          .from_address(desc.value), dtype=_cabi.STATE_DESC_DTYPE)
        stag = self._staging(D, d, W, staging)
        for r in D:
            U, Upad, eo, go = int(r["U"]), int(r["Upad"]), int(r["entry_off"]), int(r["g_off"])
            assert Upad % 4 == 0 and Upad >= U and Upad <= max_Upad
            c, l, gsrc = self._expand_state(r, d, W, stag, smin, smax, orders)
            cell_blk = _arr(cell.value + 4 * eo, W * Upad, ctypes.c_int32).reshape(W, Upad)
            cell_blk[:] = 0
            cell_blk[:, :U] = c
            for k in range(d):
                lam_blk = _arr(lam.value + 8 * (k * lam_plane + eo), W * Upad,
                               ctypes.c_double).reshape(W, Upad)
                lam_blk[:] = 0
                lam_blk[:, :U] = l[k]
            if g_per_w:
                g_blk = _arr(g.value + 8 * go, W * Upad, ctypes.c_double).reshape(W, Upad)
                g_blk[:] = 0
                g_blk[:, :U] = gsrc
            else:
                g_blk = _arr(g.value + 8 * go, Upad, ctypes.c_double)
                g_blk[:] = 0
                g_blk[:U] = gsrc[0]
        self.launches += 1
        return 0

    def sdp_build_tables_tiled(self, gref, W, g_per_w, n_states, desc, staging, n_tiles, tile_off,
                               tile_g_off, tile_U, max_tile_U, cell, lam, lam_plane, g, stream):
        d, smin, smax, orders = _grid(gref)
        D = np.frombuffer((ctypes.c_uint8 * (n_states * _cabi.STATE_DESC_DTYPE.itemsize))
                          .from_address(desc.value), dtype=_cabi.STATE_DESC_DTYPE)
        stag = self._staging(D, d, W, staging)
        toff = _arr(tile_off, n_tiles, ctypes.c_int64)
        tgoff = _arr(tile_g_off, n_tiles, ctypes.c_int64)
        tU = _arr(tile_U, n_tiles, ctypes.c_int32)
        assert n_states <= 32 * n_tiles
        for t in range(n_tiles):
            Ut = int(tU[t])
            assert Ut <= max_tile_U
            cell_blk = _arr(cell.value + 4 * int(toff[t]), Ut * W * 32, ctypes.c_int32).reshape(Ut, W, 32)
            cell_blk[:] = 0
            lam_blk = [_arr(lam.value + 8 * (k * lam_plane + int(toff[t])), Ut * W * 32,
                            ctypes.c_double).reshape(Ut, W, 32) for k in range(d)]
            for k in range(d):
                lam_blk[k][:] = 0
            if g_per_w:
                g_blk = _arr(g.value + 8 * int(toff[t]), Ut * W * 32, ctypes.c_double).reshape(Ut, W, 32)
            else:
                g_blk = _arr(g.value + 8 * int(tgoff[t]), Ut * 32, ctypes.c_double).reshape(Ut, 32)
            g_blk[:] = 0
            for lane in range(32):
                i = 32 * t + lane
                if i >= n_states:
                    break
                r = D[i]
                U = int(r["U"])
                assert U <= Ut
                c, l, gsrc = self._expand_state(r, d, W, stag, smin, smax, orders)
                cell_blk[:U, :, lane] = c.T
                for k in range(d):
                    lam_blk[k][:U, :, lane] = l[k].T
                if g_per_w:
                    g_blk[:U, :, lane] = gsrc.T
                else:
                    g_blk[:U, lane] = gsrc[0]
        self.launches += 1
        return 0

    # -- factored layouts: the model expands them to what the dense tables hold --
    def _part(self, r, d, mask, stag, smin, smax, orders, strides, n, along_u):
        """partial cell index + weights of the coordinates in `mask` for the n
        entries along the control (along_u) or perturbation axis of state r"""
        cell = np.zeros(n, dtype=np.int64)
        lams = []
        for k in range(d):
            if not (mask >> k) & 1:
                continue
            if along_u:
                idx = self._src_index(r, k, n, 1)[0]
            else:
                idx = self._src_index(r, k, 1, n)[:, 0]
            full = np.zeros((d, n))
            full[k] = stag[idx]
            # 1-D cell search on axis k alone
            ck, lk = oc.cell_search(smin[k:k + 1], smax[k:k + 1], orders[k:k + 1], full[k:k + 1])
            cell += ck.astype(np.int64) * strides[k]
            lams.append(lk[0])
        return cell, lams

    def sdp_build_tables_factored(self, gref, W, u_mask, n_states, desc, staging, cell, lam, lam_plane,
                                  g, max_Upad, cell_w, lam_w, lam_w_plane, stream):
        d, smin, smax, orders = _grid(gref)
        strides = np.concatenate([np.cumprod(orders[::-1])[::-1][1:], [1]]).astype(np.int64)
        D = np.frombuffer((ctypes.c_uint8 * (n_states * _cabi.STATE_DESC_DTYPE.itemsize))
                          .from_address(desc.value), dtype=_cabi.STATE_DESC_DTYPE)
        stag = self._staging(D, d, W, staging)
        w_mask = ~u_mask & ((1 << d) - 1)
        for i, r in enumerate(D):
            U, Upad, eo = int(r["U"]), int(r["Upad"]), int(r["entry_off"])
            assert Upad % 4 == 0 and U <= Upad <= max_Upad
            cu, lu = self._part(r, d, u_mask, stag, smin, smax, orders, strides, U, True)
            blk = _arr(cell.value + 4 * eo, Upad, ctypes.c_int32)
            blk[:] = 0
            blk[:U] = cu
            for j, l in enumerate(lu):
                blk = _arr(lam.value + 8 * (j * lam_plane + eo), Upad, ctypes.c_double)
                blk[:] = 0
                blk[:U] = l
            blk = _arr(g.value + 8 * eo, Upad, ctypes.c_double)
            blk[:] = 0
            blk[:U] = stag[self._src_index(r, d, U, 1)[0]]
            cw, lw = self._part(r, d, w_mask, stag, smin, smax, orders, strides, W, False)
            _arr(cell_w.value + 4 * i * W, W, ctypes.c_int32)[:] = cw
            for j, l in enumerate(lw):
                _arr(lam_w.value + 8 * (j * lam_w_plane + i * W), W, ctypes.c_double)[:] = l
        self.launches += 1
        return 0

    def sdp_build_tables_factored_tiled(self, gref, W, u_mask, n_states, desc, staging, n_tiles, tile_off,
                                        tile_U, max_tile_U, cell, lam, lam_plane, g, cell_w, lam_w,
                                        lam_w_plane, stream):
        d, smin, smax, orders = _grid(gref)
        strides = np.concatenate([np.cumprod(orders[::-1])[::-1][1:], [1]]).astype(np.int64)
        D = np.frombuffer((ctypes.c_uint8 * (n_states * _cabi.STATE_DESC_DTYPE.itemsize))
                          .from_address(desc.value), dtype=_cabi.STATE_DESC_DTYPE)
        stag = self._staging(D, d, W, staging)
        toff = _arr(tile_off, n_tiles, ctypes.c_int64)
        tU = _arr(tile_U, n_tiles, ctypes.c_int32)
        w_mask = ~u_mask & ((1 << d) - 1)
        n_u = bin(u_mask).count("1")
        for t in range(n_tiles):
            Ut = int(tU[t])
            assert Ut <= max_tile_U
            cblk = _arr(cell.value + 4 * int(toff[t]), Ut * 32, ctypes.c_int32).reshape(Ut, 32)
            lblk = [_arr(lam.value + 8 * (j * lam_plane + int(toff[t])), Ut * 32, ctypes.c_double).reshape(Ut, 32)
                    for j in range(n_u)]
            gblk = _arr(g.value + 8 * int(toff[t]), Ut * 32, ctypes.c_double).reshape(Ut, 32)
            cblk[:] = 0
            gblk[:] = 0
            for l in lblk:
                l[:] = 0
            cwb = _arr(cell_w.value + 4 * t * W * 32, W * 32, ctypes.c_int32).reshape(W, 32)
            lwb = [_arr(lam_w.value + 8 * (j * lam_w_plane + t * W * 32), W * 32, ctypes.c_double).reshape(W, 32)
                   for j in range(d - n_u)]
            cwb[:] = 0
            for l in lwb:
                l[:] = 0
            for lane in range(32):
                i = 32 * t + lane
                if i >= n_states:
                    break
                r = D[i]
                U = int(r["U"])
                cu, lu = self._part(r, d, u_mask, stag, smin, smax, orders, strides, U, True)
                cblk[:U, lane] = cu
                for j, l in enumerate(lu):
                    lblk[j][:U, lane] = l
                gblk[:U, lane] = stag[self._src_index(r, d, U, 1)[0]]
                cw, lw = self._part(r, d, w_mask, stag, smin, smax, orders, strides, W, False)
                cwb[:, lane] = cw
                for j, l in enumerate(lw):
                    lwb[j][:, lane] = l
        self.launches += 1
        return 0

    def _merge(self, T, d, lu, lw):
        out, ju, jw = [], 0, 0
        for k in range(d):
            if (T.u_mask >> k) & 1:
                out.append(lu[ju])
                ju += 1
            else:
                out.append(lw[jw])
                jw += 1
        return out

    def sdp_sweep(self, gref, tref, J_prev, part_val, part_idx, J_out, argmin_out, stream):
        self.sdp_sweep_partials(gref, tref, J_prev, part_val, part_idx, stream)
        return self.sdp_sweep_finalize(tref, part_val, part_idx, J_out, argmin_out, stream)

    def sdp_column_table(self, gref, tref, J_prev, stream):
        T = tref._obj
        assert T.layout == _cabi.LAYOUT_COLUMN_FACTORED and T.col_table and T.run_end and T.seg_begin
        self.col_table_J = _arr(J_prev, int(np.prod(_grid(gref)[3])), ctypes.c_double).copy()
        self.launches += 1
        return 0

    def sdp_sweep_partials(self, gref, tref, J_prev, part_val, part_idx, stream):
        d, smin, smax, orders = _grid(gref)
        T = tref._obj
        n_grid = int(np.prod(orders))
        J = _arr(J_prev, n_grid, ctypes.c_double)
        strides = np.concatenate([np.cumprod(orders[::-1])[::-1][1:], [1]]).astype(np.int64)
        items = np.frombuffer((ctypes.c_uint8 * (T.n_items * _cabi.ITEM_DTYPE.itemsize))
                              .from_address(T.items), dtype=_cabi.ITEM_DTYPE)
        p = _arr(T.p, T.W, ctypes.c_double) if T.expect else np.ones(T.W)
        column = T.layout == _cabi.LAYOUT_COLUMN_FACTORED
        tiled = column or T.layout in (_cabi.LAYOUT_STATE_MINOR, _cabi.LAYOUT_STATE_MINOR_FACTORED)
        factored = column or T.layout in (_cabi.LAYOUT_CONTROL_MINOR_FACTORED, _cabi.LAYOUT_STATE_MINOR_FACTORED)
        n_u = bin(T.u_mask).count("1")
        width = 32 if tiled else 1
        pv = _arr(part_val, T.n_items * width, ctypes.c_double)
        pi = _arr(part_idx, T.n_items * width, ctypes.c_int32)
        W = T.W
        n_pos = T.n_states        # entries of U: states, or (layout CF) positions incl. padding lanes
        if column:
            assert T.u_mask == 1 and T.n_states % T.n_cols == 0
            n_pos = (int(items["state"].max()) + 1) * 32 if len(items) else 0
            # every CTA segment is a run of the item list (this launch may cover only a part of it)
            seg = _arr(T.seg_begin, T.n_segs + 1, ctypes.c_int64)
            assert 0 <= seg[0] and seg[-1] <= T.n_items and np.all(np.diff(seg) >= 0)
            assert np.all(np.diff(items["state"]) >= 0)          # ordered by tile
            if T.col_pairs:
                assert T.item_order and T.pos_row and T.tiles_per_col % 2 == 0
            assert T.col_table and T.col_table % 16 == 0         # scratch for the column tables
            if T.col_table_ready:
                # the caller ran the pre-pass (sdp_column_table) on this J
                assert np.array_equal(self.col_table_J.view(np.int64), J.view(np.int64))
        Us = _arr(T.U, n_pos, ctypes.c_int32)

        def lerp(c, lam):
            def rec(base, k):
                if k == d:
                    return J[base]
                a = rec(base, k + 1)
                b = rec(base + strides[k], k + 1)
                return (1 - lam[k]) * a + lam[k] * b
            return rec(c, 0)

        def first_min(acc):
            nan = np.isnan(acc)
            return int(np.argmax(nan)) if nan.any() else int(np.argmin(acc))

        if column:
            self._column_partials(T, d, J, strides, orders, items, p, pv, pi, Us)
        for n_it, it in enumerate(items):
            cnt, ub = int(it["u_count"]), int(it["u_begin"])
            if column:
                continue
            if factored and not tiled:
                eb, sidx = int(it["entry_base"]), int(it["state"])
                assert int(it["g_base"]) == eb
                cu = _arr(T.cell + 4 * eb, cnt, ctypes.c_int32).astype(np.int64)
                lu = [_arr(T.lam + 8 * (j * T.lam_plane + eb), cnt, ctypes.c_double) for j in range(n_u)]
                gv = _arr(T.g + 8 * eb, cnt, ctypes.c_double)
                acc = np.zeros(cnt)
                for w in range(W):
                    f = sidx * W + w
                    cw = int(_arr(T.cell_w + 4 * f, 1, ctypes.c_int32)[0])
                    lw = [_arr(T.lam_w + 8 * (j * T.lam_w_plane + f), 1, ctypes.c_double)[0]
                          for j in range(d - n_u)]
                    jg = gv + lerp(cu + cw, self._merge(T, d, lu, lw))
                    acc = acc + jg * p[w] if T.expect else jg
                j = first_min(acc)
                pv[n_it], pi[n_it] = acc[j], ub + j
            elif factored:
                eb, tix = int(it["entry_base"]), int(it["state"])
                assert int(it["g_base"]) == eb
                cu = _arr(T.cell + 4 * eb, cnt * 32, ctypes.c_int32).astype(np.int64).reshape(cnt, 32)
                lu = [_arr(T.lam + 8 * (j * T.lam_plane + eb), cnt * 32, ctypes.c_double).reshape(cnt, 32)
                      for j in range(n_u)]
                Gv = _arr(T.g + 8 * eb, cnt * 32, ctypes.c_double).reshape(cnt, 32)
                acc = np.zeros((cnt, 32))
                for w in range(W):
                    f = (tix * W + w) * 32
                    if column:
                        # the kernel reads the column's w-part at lane 0 of its first tile
                        f0 = ((tix // T.tiles_per_col) * T.tiles_per_col * W + w) * 32
                        cw = _arr(T.cell_w + 4 * f0, 1, ctypes.c_int32).astype(np.int64)[None, :]
                        lw = [_arr(T.lam_w + 8 * (j * T.lam_w_plane + f0), 1, ctypes.c_double)[None, :]
                              for j in range(d - n_u)]
                    else:
                        cw = _arr(T.cell_w + 4 * f, 32, ctypes.c_int32).astype(np.int64)[None, :]
                        lw = [_arr(T.lam_w + 8 * (j * T.lam_w_plane + f), 32, ctypes.c_double)[None, :]
                              for j in range(d - n_u)]
                    jg = Gv + lerp(cu + cw, self._merge(T, d, lu, lw))
                    acc = acc + jg * p[w] if T.expect else jg
                for lane in range(32):
                    s_i = tix * 32 + lane
                    n_ok = max(0, min(cnt, (int(Us[s_i]) if s_i < n_pos else 0) - ub))
                    if n_ok == 0:
                        pv[n_it * 32 + lane], pi[n_it * 32 + lane] = np.inf, 2 ** 31 - 1
                    else:
                        j = first_min(acc[:n_ok, lane])
                        pv[n_it * 32 + lane], pi[n_it * 32 + lane] = acc[j, lane], ub + j
            elif not tiled:
                Upad = int(it["Upad"])
                acc = np.zeros(cnt)
                for w in range(W):
                    off = int(it["entry_base"]) + w * Upad
                    c = _arr(T.cell + 4 * off, cnt, ctypes.c_int32).astype(np.int64)
                    lam = [_arr(T.lam + 8 * (k * T.lam_plane + off), cnt, ctypes.c_double) for k in range(d)]
                    if T.g_per_w:
                        gv = _arr(T.g + 8 * (int(it["g_base"]) + w * Upad), cnt, ctypes.c_double)
                    else:
                        gv = _arr(T.g + 8 * int(it["g_base"]), cnt, ctypes.c_double)
                    jg = gv + lerp(c, lam)
                    acc = acc + jg * p[w] if T.expect else jg
                j = first_min(acc)
                pv[n_it], pi[n_it] = acc[j], ub + j
            else:
                eb = int(it["entry_base"])
                C = _arr(T.cell + 4 * eb, cnt * W * 32, ctypes.c_int32).astype(np.int64).reshape(cnt, W, 32)
                L = [_arr(T.lam + 8 * (k * T.lam_plane + eb), cnt * W * 32, ctypes.c_double).reshape(cnt, W, 32)
                     for k in range(d)]
                if T.g_per_w:
                    Gv = _arr(T.g + 8 * int(it["g_base"]), cnt * W * 32, ctypes.c_double).reshape(cnt, W, 32)
                else:
                    Gv = _arr(T.g + 8 * int(it["g_base"]), cnt * 32, ctypes.c_double).reshape(cnt, 1, 32)
                acc = np.zeros((cnt, 32))
                for w in range(W):
                    jg = Gv[:, w if T.g_per_w else 0, :] + lerp(C[:, w, :], [l[:, w, :] for l in L])
                    acc = acc + jg * p[w] if T.expect else jg
                for lane in range(32):
                    s_i = int(it["state"]) * 32 + lane
                    n_ok = max(0, min(cnt, (int(Us[s_i]) if s_i < T.n_states else 0) - ub))
                    if n_ok == 0:
                        pv[n_it * 32 + lane], pi[n_it * 32 + lane] = np.inf, 2 ** 31 - 1
                    else:
                        j = first_min(acc[:n_ok, lane])
                        pv[n_it * 32 + lane], pi[n_it * 32 + lane] = acc[j, lane], ub + j
        self.launches += 1
        return 0

    def sdp_sweep_finalize(self, tref, part_val, part_idx, J_out, argmin_out, stream):
        T = tref._obj
        column = T.layout == _cabi.LAYOUT_COLUMN_FACTORED
        tiled = column or T.layout in (_cabi.LAYOUT_STATE_MINOR, _cabi.LAYOUT_STATE_MINOR_FACTORED)
        width = 32 if tiled else 1
        n_units = (T.n_states + 31) // 32 if tiled else T.n_states
        if column:
            # one band of whole rows: n_states, tiles_per_col and item_begin are the band's
            assert T.n_states % T.n_cols == 0
            n_units = T.n_cols * T.tiles_per_col
            row_pos = None
            if T.pos_row:
                # two rows per lane: positions are not rows (pos_row: position -> row, -1 padding)
                pr = _arr(T.pos_row, T.tiles_per_col * 32, ctypes.c_int32)
                row_pos = {int(r): p_ for p_, r in enumerate(pr) if r >= 0}
                assert sorted(row_pos) == list(range(T.n_states // T.n_cols))
            else:
                assert T.tiles_per_col == (T.n_states // T.n_cols + 31) // 32
        ib = _arr(T.item_begin, n_units + 1, ctypes.c_int64)
        top = int(ib[-1]) * width
        pv = _arr(part_val, top, ctypes.c_double)
        pi = _arr(part_idx, top, ctypes.c_int32)
        Jo = _arr(J_out, T.n_states, ctypes.c_double)
        ao = _arr(argmin_out, T.n_states, ctypes.c_int32)
        for i in range(T.n_states):
            bv, bi = np.inf, 2 ** 31 - 1
            unit, lane = (i // 32, i % 32) if tiled else (i, 0)
            if column:
                row, c = divmod(i, T.n_cols)
                if row_pos is not None:
                    row = row_pos[row]
                unit, lane = c * T.tiles_per_col + row // 32, row % 32
            for k in range(ib[unit], ib[unit + 1]):
                kk = k * width + lane
                if _better(pv[kk], int(pi[kk]), bv, bi):
                    bv, bi = pv[kk], int(pi[kk])
            Jo[i], ao[i] = bv, bi
        self.launches += 1
        return 0

    def sdp_sweep_finalize_cols(self, tref, part_val, part_idx, J_out, argmin_out, glob_cols, col_begin,
                                nc, lo, hi, npts, pol, beside_sweep, stream):
        """the combine of a view on the columns [col_begin, col_begin + n_cols): results in grid
        order into whole-grid arrays; nc > 0: the control values too"""
        T = tref._obj
        assert T.layout == _cabi.LAYOUT_COLUMN_FACTORED and T.n_states % T.n_cols == 0
        assert 0 <= col_begin and col_begin + T.n_cols <= glob_cols
        n_rows = T.n_states // T.n_cols
        J_loc = np.zeros(T.n_states)
        a_loc = np.zeros(T.n_states, dtype=np.int32)
        rc = self.sdp_sweep_finalize(tref, part_val, part_idx, ctypes.c_void_p(J_loc.ctypes.data),
                                     ctypes.c_void_p(a_loc.ctypes.data), stream)
        if rc:
            return rc
        n_all = n_rows * glob_cols
        Jo = _arr(J_out, n_all, ctypes.c_double).reshape(n_rows, glob_cols)
        ao = _arr(argmin_out, n_all, ctypes.c_int32).reshape(n_rows, glob_cols)
        Jo[:, col_begin:col_begin + T.n_cols] = J_loc.reshape(n_rows, T.n_cols)
        ao[:, col_begin:col_begin + T.n_cols] = a_loc.reshape(n_rows, T.n_cols)
        if nc > 0:
            g = (np.arange(n_rows)[:, None] * glob_cols + col_begin + np.arange(T.n_cols)[None, :]).reshape(-1)
            LO = _arr(lo, n_all * nc, ctypes.c_double).reshape(n_all, nc)[g].copy()
            HI = _arr(hi, n_all * nc, ctypes.c_double).reshape(n_all, nc)[g].copy()
            NP = _arr(npts, n_all * nc, ctypes.c_int32).reshape(n_all, nc)[g].copy()
            out = np.zeros((len(g), nc))
            self.sdp_policy_values(len(g), nc, ctypes.c_void_p(LO.ctypes.data), ctypes.c_void_p(HI.ctypes.data),
                                   ctypes.c_void_p(NP.ctypes.data), ctypes.c_void_p(a_loc.ctypes.data),
                                   ctypes.c_void_p(out.ctypes.data), stream)
            _arr(pol, n_all * nc, ctypes.c_double).reshape(n_all, nc)[g] = out
        return 0

    def sdp_memcpy_2d(self, dst, dpitch, src, spitch, width, height, stream):
        assert dpitch >= width and spitch >= width
        if width and height:
            S = _arr(src, (height - 1) * spitch + width, ctypes.c_uint8)
            D = _arr(dst, (height - 1) * dpitch + width, ctypes.c_uint8)
            for r in range(height):
                D[r * dpitch:r * dpitch + width] = S[r * spitch:r * spitch + width]
        return 0

    def _column_partials(self, T, d, J, strides, orders, items, p, pv, pi, Us):
        """layout CF the way k_sweep_fact_column does it: one CTA per segment of the item
        list; at every column change the table R[row][w] = inner interpolation over the axes
        1..d-1 is rebuilt from the w-part of lane 0 of the column's first tile; a backup is
        (1-l0)*R[q0][w] + l0*R[q0+1][w] with q0 = cell_u / stride0"""
        W, Tc = T.W, T.tiles_per_col          # (tiles per column of the FIRST band)
        seg = _arr(T.seg_begin, T.n_segs + 1, ctypes.c_int64)
        n_work = int(seg[-1])           # (positions of the walking order covered by this launch)
        run_end = _arr(T.run_end, n_work, ctypes.c_int64)
        # positions -> items (SdpTables.item_order), identity when absent; with two rows per lane
        # the order lists the items of the first tile of every pair, item.g_base = the partner
        order = _arr(T.item_order, n_work, ctypes.c_int64) if T.item_order else np.arange(T.n_items)
        rows, stride0 = int(orders[0]), int(strides[0])
        P = W | 1
        done = np.zeros(len(items), dtype=bool)
        for b in range(T.n_segs):
            i, seg_end = int(seg[b]), int(seg[b + 1])
            while i < seg_end:
                col = int(items[order[i]]["Upad"])       # layout CF: the column of the item's tile
                e = min(int(run_end[i]), seg_end)
                R = np.full(rows * P + 9, np.nan)
                for w in range(W):
                    f = (col * Tc * W + w) * 32
                    cw = int(_arr(T.cell_w + 4 * f, 1, ctypes.c_int32)[0])
                    lw = [_arr(T.lam_w + 8 * (j * T.lam_w_plane + f), 1, ctypes.c_double)[0]
                          for j in range(d - 1)]

                    def rec(base, k):
                        if k == d:
                            return J[base]
                        a = rec(base, k + 1)
                        bb = rec(base + strides[k], k + 1)
                        return (1 - lw[k - 1]) * a + lw[k - 1] * bb
                    R[np.arange(rows) * P + w] = rec(np.arange(rows, dtype=np.int64) * stride0 + cw, 1)
                todo = []
                for pos in range(i, e):
                    a = int(order[pos])
                    todo.append(a)
                    if T.col_pairs:
                        b_ = int(items[a]["g_base"])
                        assert int(items[a]["state"]) % 2 == 0
                        if b_ >= 0:
                            assert (int(items[b_]["state"]) == int(items[a]["state"]) + 1
                                    and items[b_]["u_begin"] == items[a]["u_begin"]
                                    and items[b_]["u_count"] == items[a]["u_count"])
                            todo.append(b_)
                for n_it in todo:
                    it = items[n_it]
                    assert int(it["Upad"]) == col and not done[n_it]
                    done[n_it] = True
                    cnt, ub, eb, tix = int(it["u_count"]), int(it["u_begin"]), int(it["entry_base"]), int(it["state"])
                    assert T.col_pairs or int(it["g_base"]) == eb
                    cu = _arr(T.cell + 4 * eb, cnt * 32, ctypes.c_int32).astype(np.int64).reshape(cnt, 32)
                    lu = _arr(T.lam + 8 * eb, cnt * 32, ctypes.c_double).reshape(cnt, 32)
                    Gv = _arr(T.g + 8 * eb, cnt * 32, ctypes.c_double).reshape(cnt, 32)
                    assert np.all(cu % stride0 == 0)
                    q = cu // stride0
                    acc = np.zeros((cnt, 32))
                    for w in range(W):
                        v = (1 - lu) * R[q * P + w] + lu * R[q * P + P + w]
                        jg = Gv + v
                        acc = acc + jg * p[w] if T.expect else jg
                    for lane in range(32):
                        n_ok = max(0, min(cnt, int(Us[tix * 32 + lane]) - ub))
                        if n_ok == 0:
                            pv[n_it * 32 + lane], pi[n_it * 32 + lane] = np.inf, 2 ** 31 - 1
                        else:
                            a = acc[:n_ok, lane]
                            nan = np.isnan(a)
                            j = int(np.argmax(nan)) if nan.any() else int(np.argmin(a))
                            pv[n_it * 32 + lane], pi[n_it * 32 + lane] = a[j], ub + j
                i = e
        # every item the covered positions stand for was processed (with pairs: partners too)
        covered = [int(order[pos]) for pos in range(int(seg[0]), int(seg[-1]))]
        assert done[covered].all() and (T.col_pairs or done.sum() == len(covered))

    def sdp_policy_eval(self, gref, W, g_per_w, p, cell, lam, lam_plane, g, n_states, state_begin,
                        n_grid, J_a, J_b, n_iter, rel_dp, ref_index, hist, stream):
        d, smin, smax, orders = _grid(gref)
        strides = np.concatenate([np.cumprod(orders[::-1])[::-1][1:], [1]]).astype(np.int64)
        P = _arr(p, W, ctypes.c_double)
        C = _arr(cell, W * n_states, ctypes.c_int32).astype(np.int64).reshape(W, n_states)
        L = [_arr(lam.value + 8 * k * lam_plane, W * n_states, ctypes.c_double).reshape(W, n_states)
             for k in range(d)]
        Gv = _arr(g, (W if g_per_w else 1) * n_states, ctypes.c_double).reshape(-1, n_states)
        A, B = _arr(J_a, n_grid, ctypes.c_double), _arr(J_b, n_grid, ctypes.c_double)
        H = _arr(hist, n_iter, ctypes.c_double) if rel_dp else None
        src, dst = A, B
        for it in range(n_iter):
            acc = np.zeros(n_states)
            for w in range(W):
                lam_w = [L[k][w] for k in range(d)]

                def rec(base, k):
                    if k == d:
                        return src[base]
                    a = rec(base, k + 1)
                    b = rec(base + strides[k], k + 1)
                    return (1 - lam_w[k]) * a + lam_w[k] * b
                acc = acc + (Gv[w if g_per_w else 0] + rec(C[w], 0)) * P[w]
            dst[state_begin:state_begin + n_states] = acc
            if rel_dp:
                H[it] = dst[ref_index]
                dst -= H[it]
            src, dst = dst, src
        self.launches += n_iter
        return 0

    # -- the exchange over peer memory (SdpPeers): every rank's buffers are plain host memory here.
    # The epoch / flag / done words are kept as the header says; a wait on a flag that is not yet
    # published raises instead of spinning (the model runs the ranks one after the other).
    @staticmethod
    def _peers(pref):
        P = pref._obj
        assert 1 <= P.world <= _cabi.SDP_MAX_PEERS and 0 <= P.rank < P.world
        assert P.epoch and P.done and all(P.flags[r] for r in range(P.world))
        return P

    @staticmethod
    def _publish(P):
        assert _arr(P.done, 1, ctypes.c_uint32)[0] == 0       # zero between launches
        ep = _arr(P.epoch, 1, ctypes.c_uint64)
        ep[0] += 1
        for q in range(P.world):
            _arr(P.flags[q], P.world, ctypes.c_uint64)[P.rank] = ep[0]

    @staticmethod
    def _wait(P, e=None):
        e = int(_arr(P.epoch, 1, ctypes.c_uint64)[0]) if e is None else e
        f = _arr(P.flags[P.rank], P.world, ctypes.c_uint64)
        if not np.all(f >= e):
            raise AssertionError("rank %d waits for epoch %d on flags %s" % (P.rank, e, list(f)))

    def _store(self, P, dest, J_loc, a_loc):
        """J_loc / a_loc (local states) -> grid states `dest` of every rank's J (and A) buffer"""
        n_grid = int(dest.max()) + 1 if len(dest) else 0
        for q in range(P.world):
            _arr(P.J[q], n_grid, ctypes.c_double)[dest] = J_loc
            if P.A[0] and a_loc is not None:
                _arr(P.A[q], n_grid, ctypes.c_int32)[dest] = a_loc

    def _local_combine(self, tref, part_val, part_idx, argmin_out):
        T = tref._obj
        J_loc = np.zeros(T.n_states)
        if T.n_states:
            rc = self.sdp_sweep_finalize(tref, part_val, part_idx, ctypes.c_void_p(J_loc.ctypes.data),
                                         argmin_out, None)
            assert rc == 0
        return J_loc, _arr(argmin_out, T.n_states, ctypes.c_int32).copy()

    def sdp_sweep_finalize_p2p(self, tref, part_val, part_idx, argmin_out, pref, state_begin, stream):
        P = self._peers(pref)
        assert state_begin >= 0
        J_loc, a_loc = self._local_combine(tref, part_val, part_idx, argmin_out)
        self._store(P, state_begin + np.arange(len(J_loc)), J_loc, a_loc)
        self._publish(P)
        self.launches += 1
        return 0

    def sdp_sweep_finalize_p2p_cols(self, tref, part_val, part_idx, argmin_out, pref, glob_cols, col_begin,
                                    stream):
        T = tref._obj
        P = self._peers(pref)
        assert T.layout == _cabi.LAYOUT_COLUMN_FACTORED and 0 <= col_begin and col_begin + T.n_cols <= glob_cols
        J_loc, a_loc = self._local_combine(tref, part_val, part_idx, argmin_out)
        n_rows = T.n_states // T.n_cols if T.n_cols else 0
        dest = (np.arange(n_rows)[:, None] * glob_cols + col_begin + np.arange(T.n_cols)[None, :]).reshape(-1)
        self._store(P, dest, J_loc, a_loc)
        self._publish(P)
        self.launches += 1
        return 0

    def sdp_p2p_wait(self, pref, stream):
        self._wait(self._peers(pref))
        self.launches += 1
        return 0

    def sdp_sweep_partials_after(self, gref, tref, J_prev, part_val, part_idx, pref, stream):
        self._wait(self._peers(pref))
        return self.sdp_sweep_partials(gref, tref, J_prev, part_val, part_idx, stream)

    def sdp_p2p_broadcast(self, src, offset, n, pref, stream):
        P = self._peers(pref)
        assert offset >= 0 and n >= 0
        if n:
            piece = _arr(src, offset + n, ctypes.c_double)[offset:].copy()
            for q in range(P.world):
                if q != P.rank:
                    _arr(P.J[q], offset + n, ctypes.c_double)[offset:] = piece
        self._publish(P)
        self.launches += 1
        return 0

    def sdp_p2p_barrier(self, pref, stream):
        P = self._peers(pref)
        self._publish(P)
        self._wait(P)
        self.launches += 1
        return 0

    def _policy_backup(self, gref, W, g_per_w, p, cell, lam, lam_plane, g, n, J):
        """one fixed-policy backup of n states from J, in the kernel's order ([w][n] planes)"""
        d, smin, smax, orders = _grid(gref)
        strides = np.concatenate([np.cumprod(orders[::-1])[::-1][1:], [1]]).astype(np.int64)
        P = _arr(p, W, ctypes.c_double)
        C = _arr(cell, W * n, ctypes.c_int32).astype(np.int64).reshape(W, n)
        L = [_arr(lam.value + 8 * k * lam_plane, W * n, ctypes.c_double).reshape(W, n) for k in range(d)]
        Gv = _arr(g, (W if g_per_w else 1) * n, ctypes.c_double).reshape(-1, n)
        acc = np.zeros(n)
        for w in range(W):
            lam_w = [L[k][w] for k in range(d)]

            def rec(base, k):
                if k == d:
                    return J[base]
                a = rec(base, k + 1)
                b = rec(base + strides[k], k + 1)
                return (1 - lam_w[k]) * a + lam_w[k] * b
            acc = acc + (Gv[w if g_per_w else 0] + rec(C[w], 0)) * P[w]
        return acc

    def sdp_policy_eval_p2p(self, gref, W, g_per_w, p, cell, lam, lam_plane, g, n_states, state_begin, n_grid,
                            J_in, pref, ref_cell, ref_lam, ref_g, J_ref_out, stream):
        P = self._peers(pref)
        assert 0 <= state_begin and state_begin + n_states <= n_grid
        J = _arr(J_in, n_grid, ctypes.c_double)
        acc = self._policy_backup(gref, W, g_per_w, p, cell, lam, lam_plane, g, n_states, J) \
            if n_states else np.zeros(0)
        if ref_cell:
            assert ref_lam and ref_g and J_ref_out
            # the reference state's entries: [W], [d][W], [W] or [1] (stride 1, lam plane W)
            ref = self._policy_backup(gref, W, g_per_w, p, ref_cell, ref_lam, W, ref_g, 1, J)[0]
            _arr(J_ref_out, 1, ctypes.c_double)[0] = ref
            acc = acc - ref
        self._store(P, state_begin + np.arange(n_states), acc, None)
        self._publish(P)
        self.launches += 1
        return 0

    def sdp_policy_values(self, n, nc, lo, hi, npts, argmin, pol, stream):
        LO = _arr(lo, n * nc, ctypes.c_double).reshape(n, nc)
        HI = _arr(hi, n * nc, ctypes.c_double).reshape(n, nc)
        NP = _arr(npts, n * nc, ctypes.c_int32).reshape(n, nc)
        AM = _arr(argmin, n, ctypes.c_int32).astype(np.int64)
        out = _arr(pol, n * nc, ctypes.c_double).reshape(n, nc)
        for i in range(n):
            ind = np.unravel_index(AM[i], tuple(NP[i]))
            for c in range(nc):
                m = int(NP[i, c])
                grid = np.array([(LO[i, c] + HI[i, c]) / 2]) if m == 1 else np.linspace(LO[i, c], HI[i, c], m)
                out[i, c] = grid[ind[c]]
        return 0

    def sdp_rel_shift(self, J, n, ref_index, ref_out, stream):
        A = _arr(J, n, ctypes.c_double)
        r = _arr(ref_out, 1, ctypes.c_double)
        r[0] = A[ref_index]
        A -= r[0]
        return 0

    def sdp_supnorm_diff(self, a, b, n, out, stream):
        d = np.abs(_arr(a, n, ctypes.c_double) - _arr(b, n, ctypes.c_double))
        d = d[~np.isnan(d)]
        _arr(out, 1, ctypes.c_double)[0] = d.max() if d.size else 0.0
        return 0

    def sdp_interp(self, gref, n_v, values, n_s, s, out, stream):
        d, smin, smax, orders = _grid(gref)
        n_grid = int(np.prod(orders))
        V = _arr(values, n_v * n_grid, ctypes.c_double).reshape(n_v, n_grid)
        S = _arr(s, d * n_s, ctypes.c_double).reshape(d, n_s)
        _arr(out, n_v * n_s, ctypes.c_double)[:] = oc.interp(smin, smax, orders, V, S).reshape(-1)
        return 0

    def sdp_interp_f32(self, gref, n_v, values, n_s, s, out, stream):
        d, smin, smax, orders = _grid(gref)
        n_grid = int(np.prod(orders))
        V = _arr(values, n_v * n_grid, ctypes.c_float).reshape(n_v, n_grid)
        S = _arr(s, d * n_s, ctypes.c_float).reshape(d, n_s)
        _arr(out, n_v * n_s, ctypes.c_float)[:] = oc.interp(smin, smax, orders, V, S).reshape(-1)
        return 0
