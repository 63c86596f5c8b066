"""numpy twin of the path sampler (sdp_chain_pack / sdp_chain_sample of include/sdp_b200.h).

TEST AND MEASUREMENT INFRASTRUCTURE.  The same records, the same Philox-4x32-10 bits and the same
fp64 operations in the same order as the kernels, vectorised over the paths: the GPU tests
compare the kernels with it bit for bit, and the CPU tests drive the host code through it.
"""
import numpy as np

from stodynprog_b200 import _cabi

_MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox-4x32-10 on arrays of 32-bit counter words (held in uint64), key (k0, k1)"""
    c = [np.asarray(v, dtype=np.uint64) & _MASK for v in np.broadcast_arrays(c0, c1, c2, c3)]
    k0, k1 = np.uint64(k0), np.uint64(k1)
    m0, m1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
    for i in range(10):
        if i:
            k0 = (k0 + np.uint64(0x9E3779B9)) & _MASK
            k1 = (k1 + np.uint64(0xBB67AE85)) & _MASK
        p0, p1 = m0 * c[0], m1 * c[2]                  # 32 x 32 -> 64 bits, exact
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & _MASK, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & _MASK]
    return c


def u01(lo, hi):
    """the double of two words: ((lo | hi << 32) >> 11) * 2^-53"""
    return ((hi << np.uint64(32) | lo) >> np.uint64(11)).astype(np.float64) * 2.0 ** -53


def pack(d, W, g_per_w, n, cell, lam, g):
    """records [n*W][chain_rec(d)] of the planes cell [W*n], lam [d][W*n], g [W*n or n]"""
    R = _cabi.chain_rec(d)
    rec = np.zeros((n * W, R))
    rec[:, 0] = np.asarray(cell, dtype=np.int32).astype(np.uint32).astype(np.uint64).view(np.float64)
    rec[:, 1:1 + d] = np.asarray(lam, dtype=float).reshape(d, n * W).T
    g = np.asarray(g, dtype=float)
    rec[:, 1 + d] = g if g_per_w else np.tile(g[:n], W)
    return rec


def sample(strides, W, cdf, rec, n, n_steps, step0, seed, fresh, state, total, hit, counters,
           start_cdf=None, target=None, rec_steps=None, rec_out=None):
    """advance the paths in place, exactly as k_chain_sample.  state / total / hit [M];
    target: uint32 words; rec_steps: increasing global steps; rec_out [len(rec_steps)][M];
    counters [2] += (clamped, NaN transitions)"""
    d = len(strides)
    M = state.size
    k0, k1 = seed & 0xFFFFFFFF, seed >> 32
    path = np.arange(M, dtype=np.uint64)
    cdf = np.asarray(cdf, dtype=float)
    cell = rec[:, 0].copy().view(np.uint64).astype(np.uint32).view(np.int32).astype(np.int64)
    lam, g = rec[:, 1:1 + d], rec[:, 1 + d]
    if fresh:
        acc, h = np.zeros(M), np.full(M, -1, dtype=np.int64)
        if start_cdf is not None:
            r = philox4x32_10(path, _cabi.CHAIN_INIT_STEP, 0, 0, k0, k1)
            t = u01(r[0], r[1]) * start_cdf[-1]
            x = np.minimum(np.searchsorted(start_cdf, t, side="right"), n - 1)
        else:
            x = state.astype(np.int64)
    else:
        x, acc, h = state.astype(np.int64), total.copy(), hit.astype(np.int64)
    steps = list(rec_steps) if rec_steps is not None else []
    for k in range(n_steps + 1):
        s = step0 + k
        if s in steps:
            rec_out[steps.index(s)] = x
        if target is not None:
            inside = ((target[x >> 5].astype(np.int64) >> (x & 31)) & 1).astype(bool)
            h = np.where((h < 0) & inside, s, h)
        if k == n_steps:
            break
        r0 = philox4x32_10(path, s, 0, 0, k0, k1)
        v = [u01(r0[2], r0[3])]
        if d >= 2:
            r1 = philox4x32_10(path, s, 1, 0, k0, k1)
            v += [u01(r1[0], r1[1]), u01(r1[2], r1[3])]
        if d >= 4:
            r2 = philox4x32_10(path, s, 2, 0, k0, k1)
            v += [u01(r2[0], r2[1])]
        w = np.minimum(np.searchsorted(cdf, u01(r0[0], r0[1]) * cdf[-1], side="right"), W - 1)
        e = w * n + x
        y = cell[e].copy()
        clamped, nan = np.zeros(M, dtype=bool), np.zeros(M, dtype=bool)
        for kk in range(d):
            lk = lam[e, kk]
            isnan = np.isnan(lk)
            nan |= isnan
            clamped |= (lk < 0) | (lk > 1)
            y += ((~isnan) & (v[kk] < np.clip(lk, 0.0, 1.0))) * strides[kk]
        acc = acc + g[e]
        counters[0] += int(clamped.sum())
        counters[1] += int(nan.sum())
        x = y
    state[:] = x
    total[:] = acc
    hit[:] = h
