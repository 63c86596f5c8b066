"""Device side of the solver: table residency, sweep launches, collectives.

torch is plumbing here: it owns the device buffers, the stream and the
process group.  Every compute step goes through the C ABI (`_cabi`), i.e. the
hand-written sm_100a kernels in csrc/sdp_b200.cu.  There is no CPU path.

Multi-GPU model (SURVEY.md §8e): one process per GPU; the C-order flattened state
grid is cut into contiguous slabs balanced by the number of admissible
controls; each rank holds the tables of its slab only; the value function J
(8 bytes per state) is replicated.  One exchange per sweep: all-gather of the
new J slab (+ an all-reduce-max of the sup-norm residual when asked).
"""
import ctypes
import os

import numpy as np

from . import _cabi
from . import tabulate as tb
from .tablebuild import (                                        # noqa: F401  (re-exported)
    COLUMN_HOIST_DEFAULT, SLAB_AXIS_DEFAULT, COLUMN_PAIRS_DEFAULT, ITEMS_TARGET,
    BuildPlan, ShardBuild, SweepTables, fill_c_tables, partition_by_weight, rebalance_bounds,
    make_items, pick_item_chunk, host_threads, pair_positions, column_order, item_run_ends,
    column_segments, column_piece_cuts, row_aligned, ColumnHoistRefused, _ColumnsNotApplicable)

__all__ = ["Engine", "SweepTables", "PolicyTables", "partition_by_weight", "rebalance_bounds",
           "column_order", "column_segments", "row_aligned"]


def _torch():
    import torch
    return torch


class _DeviceBoundLib(object):
    """The C ABI launches on the calling thread's CURRENT device (it takes raw pointers and a
    stream, and never calls cudaSetDevice).  An Engine made for `device` must therefore make that
    device current around every entry point, or DPSolver(sys, device='cuda:1') would launch on
    GPU 0 against GPU 1 pointers.  `torch.cuda.device` is a no-op when the device is already
    current (one C++ call)."""

    def __init__(self, lib, device):
        self._lib = lib
        self._guard = _torch().cuda.device(device)
        self._wrapped = {}

    def __getattr__(self, name):
        fn = self._wrapped.get(name)
        if fn is None:
            raw = getattr(self._lib, name)
            if not name.startswith("sdp_") or name in ("sdp_version", "sdp_last_error", "sdp_launch_count",
                                                       "sdp_last_kernel", "sdp_set_option"):
                return raw
            guard = self._guard

            def fn(*args):
                with guard:
                    return raw(*args)
            self._wrapped[name] = fn
        return fn


class Collective(object):
    """Thin wrapper over torch.distributed for the per-sweep exchange.
    Works with NCCL (CUDA tensors, on the current stream) and gloo (CPU tensors,
    used by the world_size-2 host tests)."""

    def __init__(self, group=None):
        torch = _torch()
        import torch.distributed as dist
        self.dist = dist
        self.group = group
        if dist.is_available() and dist.is_initialized():
            self.world = dist.get_world_size(group)
            self.rank = dist.get_rank(group)
        else:
            self.world = 1
            self.rank = 0
        self._plans = {}

    def all_gather_object(self, obj):
        if self.world == 1:
            return [obj]
        out = [None] * self.world
        self.dist.all_gather_object(out, obj, group=self.group)
        return out

    def plan(self, bounds, device):
        """index plan for gathering uneven contiguous slabs through one padded
        all_gather_into_tensor"""
        torch = _torch()
        key = (tuple(bounds), str(device))
        if key not in self._plans:
            counts = np.diff(np.asarray(bounds))
            maxc = int(counts.max()) if len(counts) else 0
            idx = np.concatenate([r * maxc + np.arange(c) for r, c in enumerate(counts)]) \
                if maxc > 0 else np.zeros(0, dtype=np.int64)
            self._plans[key] = (maxc, torch.from_numpy(idx.astype(np.int64)).to(device))
        return self._plans[key]

    def all_gather_slabs(self, local, bounds, out=None):
        """local: 1-D tensor holding this rank's slab [bounds[rank], bounds[rank+1]).
        Returns the concatenation over ranks (length bounds[-1])."""
        torch = _torch()
        if self.world == 1:
            if out is not None:
                out.copy_(local)
                return out
            return local
        maxc, index = self.plan(bounds, local.device)
        pad_local = torch.zeros(maxc, dtype=local.dtype, device=local.device)
        pad_local[:local.numel()] = local
        pad_full = torch.empty(maxc * self.world, dtype=local.dtype, device=local.device)
        self.dist.all_gather_into_tensor(pad_full, pad_local, group=self.group)
        if out is not None:
            torch.index_select(pad_full, 0, index, out=out)
            return out
        return pad_full.index_select(0, index)

    def all_gather_indexed(self, local, maxc, index, out=None):
        """all-gather of unequal 1-D pieces followed by one index_select: element g of the
        result is element index[g] of the rank-major padded concatenation (rank r's piece at
        [r*maxc, r*maxc + len)).  Used when the pieces are not contiguous slabs of the
        result (grid sharded by columns)."""
        torch = _torch()
        if self.world == 1:
            res = local.index_select(0, index)
            if out is not None:
                out.copy_(res)
                return out
            return res
        pad_local = torch.zeros(maxc, dtype=local.dtype, device=local.device)
        pad_local[:local.numel()] = local
        pad_full = torch.empty(maxc * self.world, dtype=local.dtype, device=local.device)
        self.dist.all_gather_into_tensor(pad_full, pad_local, group=self.group)
        if out is not None:
            torch.index_select(pad_full, 0, index, out=out)
            return out
        return pad_full.index_select(0, index)

    def all_reduce_max(self, t):
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX, group=self.group)
        return t

    def barrier(self):
        if self.world > 1:
            self.dist.barrier(group=self.group)


class PeerExchange(object):
    """Symmetric (peer-mapped) J double buffer + flag words for the fused
    combine + all-gather of the sweep (`sdp_sweep_finalize_p2p`): every rank's
    combine kernel stores its slab of the new J straight into every rank's
    buffer over NVLink and publishes an epoch; consumers wait on local flags.

    Buffer protocol (ping-pong): a sweep reads J[k] and writes J[1-k] on all
    ranks; the per-sweep wait guarantees that a rank can only be one sweep ahead
    of its peers, so the buffer it writes is never one a peer still reads.
    `barrier()` must separate public calls (a peer may still be copying the last
    result out of the buffer the next call will write)."""

    def __init__(self, engine, n_grid):
        import torch
        import torch.distributed._symmetric_memory as symm
        coll = engine.coll
        self.engine = engine
        self.n_grid = n_grid
        world, rank = coll.world, coll.rank
        if world > _cabi.SDP_MAX_PEERS:
            raise ValueError("peer exchange supports at most %d ranks" % _cabi.SDP_MAX_PEERS)
        group = coll.group if coll.group is not None else coll.dist.group.WORLD
        n_pad = (n_grid + 31) // 32 * 32
        # [J0 | J1 | flags (world u64, padded to 32 words)]
        self.buf = symm.empty(2 * n_pad + 32, dtype=torch.float64, device=engine.device)
        self.buf.zero_()
        self.hdl = symm.rendezvous(self.buf, group)
        torch.cuda.synchronize(engine.device)
        self.hdl.barrier()                      # zeros visible everywhere before first use
        self.n_pad = n_pad
        self._views = {}
        self.J = [self.buf[:n_grid], self.buf[n_pad:n_pad + n_grid]]
        self.local = torch.zeros(4, dtype=torch.int64, device=engine.device)   # [epoch, done]
        # every rank's full-grid argmin, filled by the peers' combine kernels like J (SdpPeers.A)
        self.abuf = symm.empty(n_pad, dtype=torch.int32, device=engine.device)
        self.abuf.zero_()
        self.ahdl = symm.rendezvous(self.abuf, group)
        torch.cuda.synchronize(engine.device)
        self.ahdl.barrier()
        self.argmin = self.abuf[:n_grid]
        aptrs = [int(p) for p in self.ahdl.buffer_ptrs]
        ptrs = [int(p) for p in self.hdl.buffer_ptrs]
        self.peers = []
        self.peers_J_only = []      # the same exchanges without the argmin (sweeps of a device-resident loop)
        for with_argmin in (True, False):
            for k in range(2):
                P = _cabi.SdpPeers()
                P.world, P.rank = world, rank
                for r in range(world):
                    P.J[r] = ptrs[r] + 8 * k * n_pad
                    P.flags[r] = ptrs[r] + 8 * 2 * n_pad
                    P.A[r] = aptrs[r] if with_argmin else None
                P.epoch = self.local.data_ptr()
                P.done = self.local.data_ptr() + 8
                (self.peers if with_argmin else self.peers_J_only).append(P)

    def peer_view(self, r, k):
        """rank r's copy of J buffer k as a tensor on this device (peer-mapped)"""
        import torch
        key = (r, k)
        if key not in self._views:
            self._views[key] = self.hdl.get_buffer(r, (self.n_grid,), torch.float64, k * self.n_pad)
        return self._views[key]

    def index_of(self, t):
        """0/1 when `t` is one of the two J buffers, else None"""
        for k in range(2):
            if t.data_ptr() == self.J[k].data_ptr() and t.numel() == self.n_grid:
                return k
        return None

    def barrier(self):
        eng = self.engine
        rc = eng.lib.sdp_p2p_barrier(ctypes.byref(self.peers[0]), eng.stream)
        _cabi.check(rc, "sdp_p2p_barrier")


class PolicyTables(object):
    """[w][n_states] planes for the fixed-policy backup (eval_policy)."""

    def __init__(self):
        self.grid = None
        self.W = 1
        self.g_per_w = 0
        self.cell = self.lam = self.g = self.p = None
        self.ref_cell = self.ref_lam = self.ref_g = None   # reference state's entries (several ranks)
        self.lam_plane = 0
        self.state_begin = 0
        self.n_states = 0
        self.bounds = None


class ChainTables(object):
    """The path sampler's tables of a fixed policy (sdp_chain_*): packed (x, w) records, device
    fp64 [n*W*chain_rec(d)], and the cumulative node probabilities, device fp64 [W]."""

    def __init__(self):
        self.grid = None
        self.W = 1
        self.n = 0
        self.rec = self.cdf = None


class Engine(object):
    """Owns the device, the stream, the process group and the launches."""

    def __init__(self, device=None, group=None, item_chunk=None, _test_lib=None):
        torch = _torch()
        self.coll = Collective(group)
        # controls per work item (one warp each).  None = adaptive: 512, halved while the
        # slab yields fewer warps than a few waves of the machine (small grids, or
        # one slab of a grid cut over 8 GPUs), see build_sweep_tables
        self.item_chunk_auto = not item_chunk
        self.item_chunk = int(item_chunk) if item_chunk else 512
        if self.item_chunk % 4:
            raise ValueError("item_chunk must be a multiple of 4")
        if _test_lib is not None:
            # TEST SEAM ONLY (tests/fake_lib.py): a numpy model of the C ABI used to
            # exercise the host logic (descriptors, items, slabs, collectives) on a
            # machine without a GPU.  Never set by the package itself.
            self.lib = _test_lib
            self.device = torch.device("cpu")
            self._cuda = False
            self._peer = {}
            self._grid_cache = {}
            self._scan_cache = None
            return
        self._peer = {}                          # n_grid -> PeerExchange | None
        self._grid_cache = {}
        self._scan_cache = None
        self.lib = _cabi.load_library()          # raises if the extension is missing
        if not torch.cuda.is_available():
            raise _cabi.SdpLibraryError(
                "no CUDA device visible: stodynprog_b200 has no CPU path "
                "(the CPU oracle lives under oracle/ and is test infrastructure only)")
        if device is None:
            device = torch.device("cuda", torch.cuda.current_device())
        self.device = torch.device(device)
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self._cuda = True
        self.lib = _DeviceBoundLib(self.lib, self.device)

    # -- helpers ----------------------------------------------------------
    @property
    def stream(self):
        torch = _torch()
        if not self._cuda:
            return ctypes.c_void_p(0)
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    @property
    def torch_stream(self):
        """the launching stream (torch's current stream of THIS engine's device)"""
        return _torch().cuda.current_stream(self.device)

    def _ptr(self, t):
        return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)

    def to_device(self, a, dtype=None):
        torch = _torch()
        a = np.ascontiguousarray(a)
        if not a.flags.writeable:
            a = a.copy()
        t = torch.from_numpy(a)
        if dtype is not None:
            t = t.to(dtype)
        if self._cuda and t.numel() * t.element_size() >= (1 << 20):
            # large inputs go through a pinned staging buffer (async DMA)
            pin = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
            pin.copy_(t)
            return pin.to(self.device, non_blocking=True)
        return t.to(self.device, non_blocking=False)

    _TORCH_DTYPES = {"float64": "float64", "int32": "int32", "int64": "int64", "uint8": "uint8"}

    def to_device_packed(self, arrays):
        """Several host arrays -> ONE page-locked staging buffer -> one asynchronous
        H2D copy; returns the device views (same shapes and dtypes).  Table builds
        upload a dozen small arrays; one by one each is a synchronous pageable copy
        (a stream synchronisation apiece), which dominates small or time-dependent
        problems that rebuild their tables at every instant."""
        torch = _torch()
        arrs = []
        for a in arrays:
            a = np.ascontiguousarray(a)
            if a.dtype.name not in self._TORCH_DTYPES:
                a = a.view(np.uint8).reshape(-1)          # structured records travel as bytes
            arrs.append(a)
        if not self._cuda:
            return [torch.from_numpy(a.copy()) for a in arrs]
        offs, total = [], 0
        for a in arrs:
            total = (total + 15) // 16 * 16
            offs.append(total)
            total += a.nbytes
        pin = torch.empty(max(total, 16), dtype=torch.uint8, pin_memory=True)
        pn = pin.numpy()
        for a, o in zip(arrs, offs):
            if a.nbytes:
                pn[o:o + a.nbytes] = a.reshape(-1).view(np.uint8)
        buf = pin.to(self.device, non_blocking=True)
        outs = []
        for a, o in zip(arrs, offs):
            t = buf[o:o + a.nbytes].view(getattr(torch, self._TORCH_DTYPES[a.dtype.name]))
            outs.append(t.reshape(a.shape))
        return outs

    def to_device_concat(self, records, parts, threads=1):
        """a structured record array + a LIST of fp64 arrays -> one page-locked buffer -> one
        asynchronous H2D copy; returns (records as device bytes, the parts concatenated without gaps
        as one device fp64 tensor).  Each part is copied once, straight into the upload buffer
        (`threads` > 1: the large parts by that many host threads side by side)."""
        torch = _torch()
        rec = np.ascontiguousarray(records).view(np.uint8).reshape(-1)
        n_parts = int(sum(a.size for a in parts))
        off = (rec.nbytes + 15) // 16 * 16
        total = off + 8 * n_parts
        host = torch.empty(max(total, 16), dtype=torch.uint8, pin_memory=self._cuda)
        hn = host.numpy()
        hn[:rec.nbytes] = rec
        dst = hn[off:off + 8 * n_parts].view(np.float64)
        pos, jobs = 0, []
        for a in parts:
            jobs.append((pos, a.reshape(-1)))
            pos += a.size

        def copy(job):
            dst[job[0]:job[0] + job[1].size] = job[1]

        big = [j for j in jobs if j[1].size >= (1 << 17)]
        if threads > 1 and len(big) > 1:
            from concurrent.futures import ThreadPoolExecutor
            if getattr(self, "_copy_pool", None) is None or self._copy_pool._max_workers != threads:
                self._copy_pool = ThreadPoolExecutor(max_workers=threads, thread_name_prefix="sdp-stage")
            list(self._copy_pool.map(copy, big))
            jobs = [j for j in jobs if j[1].size < (1 << 17)]
        for j in jobs:
            copy(j)
        buf = host.to(self.device, non_blocking=True) if self._cuda else host
        return buf[:rec.nbytes], buf[off:off + 8 * n_parts].view(torch.float64)

    def sync(self):
        if self._cuda:
            _torch().cuda.synchronize(self.device)

    # -- J buffers / peer exchange ------------------------------------------
    def peer_exchange(self, n_grid):
        """PeerExchange for grids of n_grid points, or None (one rank, CPU test
        seam, SDP_P2P=0, or symmetric memory not available: the NCCL all-gather
        path is used instead)."""
        if n_grid not in self._peer:
            px = None
            if self._cuda and self.coll.world > 1 and os.environ.get("SDP_P2P", "1") != "0":
                try:
                    px = PeerExchange(self, n_grid)
                except Exception as e:            # no P2P / symmetric memory on this box
                    import warnings
                    warnings.warn("peer-memory exchange unavailable (%s: %s); using NCCL all-gather"
                                  % (type(e).__name__, e))
                    px = None
                # every rank must take the same path
                ok = self.coll.all_gather_object(px is not None)
                if not all(ok):
                    px = None
            self._peer[n_grid] = px
        return self._peer[n_grid]

    def host_share(self, n_grid, nc):
        """HostShare for results of [n_grid] states x nc controls, or None: one rank, no peer
        exchange (the argmin must travel with J), SDP_HOST_SHARE=0, or shared memory /
        cudaHostRegister not available - same answer on every rank"""
        key = ("host_share", n_grid, nc)
        if key not in self._peer:
            hs = None
            if (self.coll.world > 1 and self.peer_exchange(n_grid) is not None
                    and os.environ.get("SDP_HOST_SHARE", "1") != "0"):
                from .hostshare import HostShare
                err = None
                try:
                    hs = HostShare(self.coll, n_grid, nc, self._cuda)
                except Exception as e:          # every rank must still take part in the vote below
                    err = e
                ok = self.coll.all_gather_object(hs is not None)
                if not all(ok):
                    if err is not None:
                        import warnings
                        warnings.warn("shared host results unavailable (%s: %s)" % (type(err).__name__, err))
                    hs = None
            self._peer[key] = hs
        return self._peer[key]

    def sweep_shared(self, hs, T, J_next, rel_ref_index=None, want_results=True, while_waiting=None):
        """One sweep with host arrays in and out through the shared page-locked segment `hs`:
        every rank uploads 1/N of J_next and hands it to its peers over NVLink, sweeps its shard
        (the combine kernel stores J AND the argmin into every rank's buffers), maps 1/N of the
        policy to control values and copies 1/N of (J, pol) into the shared result slot over its
        own PCIe link.  Returns (J, pol, J_ref) as views of the slot (None, None, J_ref when
        `want_results` is False), or None when no slot is free (the caller takes the private-
        copy path; same decision on every rank)."""
        import time
        torch = _torch()
        world, rank = self.coll.world, self.coll.rank
        n_grid, nc = hs.n_grid, hs.nc
        px = self.peer_exchange(n_grid)
        tm = [time.perf_counter()]
        # 1. where is the input, which slot takes the output (rank 0's array decides)
        src = -2
        if rank == 0:
            src = hs.slot_of(J_next)
            if src is None:
                hs.stage_J().numpy()[:] = np.asarray(J_next, dtype=np.float64).reshape(-1)
                src = -1
        hs.publish(0, src if rank == 0 else 0)
        hs.publish(1, hs.live_mask())
        hs.barrier()
        src = hs.read(0, 0)
        live = 0
        for r in range(world):
            live |= hs.read(r, 1)
        out = next((s_ for s_ in range(hs.n_slots) if s_ != src and not (live >> s_) & 1), None)
        if out is None:
            return None
        J_src = hs.stage_J() if src < 0 else hs.slot_J(src)
        tm.append(time.perf_counter())
        # 2. upload 1/N, hand it to the peers
        # (no begin_call barrier: every rank passed the host barrier above after synchronising its
        # previous call, so nobody still touches the J buffers)
        J_prev, J_new = self.J_pair(n_grid)
        self.flush_exchange()
        a, b = n_grid * rank // world, n_grid * (rank + 1) // world
        k = px.index_of(J_prev)
        J_prev[a:b].copy_(J_src[a:b], non_blocking=True)
        rc = self.lib.sdp_p2p_broadcast(self._ptr(J_prev), a, b - a, ctypes.byref(px.peers_J_only[k]), self.stream)
        _cabi.check(rc, "sdp_p2p_broadcast")
        rc = self.lib.sdp_p2p_wait(ctypes.byref(px.peers_J_only[k]), self.stream)
        _cabi.check(rc, "sdp_p2p_wait")
        tm.append(time.perf_counter())
        # 3. the sweep; J_new and the argmin are complete on every rank after the flag wait
        ref_out = torch.zeros(1, dtype=torch.float64, device=self.device) if rel_ref_index is not None else None
        self.sweep(T, J_prev, J_new, rel_ref_index=rel_ref_index, ref_out=ref_out)
        tm.append(time.perf_counter())
        # 4. 1/N of the results -> the shared slot
        pol = torch.empty((b - a, max(nc, 1)), dtype=torch.float64, device=self.device)
        if nc and b > a:
            rc = self.lib.sdp_policy_values(
                b - a, nc, ctypes.c_void_p(T.lo_dev.data_ptr() + 8 * nc * a),
                ctypes.c_void_p(T.hi_dev.data_ptr() + 8 * nc * a),
                ctypes.c_void_p(T.npts_dev.data_ptr() + 4 * nc * a),
                ctypes.c_void_p(px.argmin.data_ptr() + 4 * a), self._ptr(pol), self.stream)
            _cabi.check(rc, "sdp_policy_values")
        hs.slot_J(out)[a:b].copy_(J_new[a:b], non_blocking=True)
        if nc:
            hs.slot_pol(out)[a * nc:b * nc].copy_(pol.view(-1)[:(b - a) * nc], non_blocking=True)
        ref_host = None
        if ref_out is not None:
            ref_host = self.host_result_buffer((1,), torch.float64)
            ref_host.copy_(ref_out, non_blocking=True)
        tm.append(time.perf_counter())
        if while_waiting is not None:
            while_waiting()
        tm.append(time.perf_counter())
        self.torch_stream.synchronize() if self._cuda else None
        tm.append(time.perf_counter())
        hs.barrier()
        tm.append(time.perf_counter())
        # host-side seconds: [agree on slots, enqueue upload + hand-over, enqueue sweep, enqueue result
        # copies, cache check, wait for the GPU, host barrier] (diagnostics, bench --shared-timing)
        self.last_shared_timing = [b_ - a_ for a_, b_ in zip(tm[:-1], tm[1:])]
        J_ref = float(ref_host[0]) if ref_host is not None else None
        if not want_results:
            return None, None, J_ref
        return hs, out, J_ref

    def J_pair(self, n_grid):
        """two device fp64 [n_grid] buffers to ping-pong sweeps between; with several
        ranks they live in symmetric memory so that the sweep's combine kernel can
        store new values directly into every rank's copy"""
        torch = _torch()
        px = self.peer_exchange(n_grid)
        if px is not None:
            return px.J[0], px.J[1]
        return (torch.empty(n_grid, dtype=torch.float64, device=self.device),
                torch.empty(n_grid, dtype=torch.float64, device=self.device))

    def begin_call(self, n_grid):
        """separate two public calls that reuse the symmetric J buffers"""
        self.flush_exchange()
        px = self._peer.get(n_grid)
        if px is not None:
            px.barrier()

    def share_J(self, J, root=0):
        """make rank `root`'s device copy of J (one of the J_pair buffers) the copy of every
        rank: peer-memory stores over NVLink + flag barrier, or an NCCL broadcast.
        Collective: every rank calls it."""
        if self.coll.world == 1:
            return
        self.flush_exchange()
        px = self._peer.get(J.numel())
        k = px.index_of(J) if px is not None else None
        if k is None:
            self.coll.dist.broadcast(J, src=root, group=self.coll.group)
            return
        if self.coll.rank == root:
            for r in range(self.coll.world):
                if r != root:
                    px.peer_view(r, k).copy_(J, non_blocking=True)
        px.barrier()

    def upload_J(self, J_host, dst):
        """host fp64 array -> device buffer `dst`, asynchronously on the current stream.

        The arrays this package returns live in page-locked memory (`to_host`), so
        the usual loop `J, pol = solver.value_iteration(J)` hands back a buffer the
        DMA engine can read directly: no staging copy.  Any other array is staged
        through a pinned buffer in a few chunks, so that the H2D of one chunk
        overlaps the host copy of the next.  Every public call synchronises the
        stream before returning, so the caller's array is never read after that."""
        torch = _torch()
        a = np.ascontiguousarray(np.asarray(J_host, dtype=np.float64).reshape(-1))
        if not self._cuda:
            dst.copy_(torch.from_numpy(a))
            return dst
        src = None
        if a.flags.writeable:
            t = torch.from_numpy(a)
            if t.is_pinned():
                src = t
        if src is not None:
            dst.copy_(src, non_blocking=True)
            return dst
        n = a.size
        pin = torch.empty(n, dtype=torch.float64, pin_memory=True)
        pin_np = pin.numpy()
        step = max((n + 3) // 4, 1 << 16)
        for b0 in range(0, n, step):
            b1 = min(b0 + step, n)
            pin_np[b0:b1] = a[b0:b1]
            dst[b0:b1].copy_(pin[b0:b1], non_blocking=True)
        return dst

    # -- slab balance -----------------------------------------------------
    REBALANCE_MIN_BACKUPS = 500 * 1000 * 1000    # "auto": only sweeps long enough to matter
    REBALANCE_TOLERANCE = 1.03                   # slowest / mean slab time that is left alone
    REBALANCE_SKEW = None                        # test hook (tests/multi_gpu_check.py)

    def _measured_bounds(self, T, U_all):
        """Slab boundaries equalising the MEASURED sweep time of the ranks.

        Cutting the grid by the number of admissible controls balances the backups,
        not the time: the cost of a backup depends on where its corners fall (L1 / L2
        hit rates differ between regions of the state space) and on the GPU (measured
        on 8 B200s, config #5: 0.375 .. 0.454 ms for slabs of equal backup count).
        Every rank times the streaming kernel on its slab; the per-state weights of a
        slab are scaled by its measured time per weight and the grid is cut again.
        Returns the new boundaries, or None when the slabs are already balanced.
        Same data on every rank (all-gathered), so every rank takes the same decision;
        results do not depend on the partition."""
        torch = _torch()
        coll = self.coll
        n_grid = len(U_all)
        J = torch.zeros(n_grid, dtype=torch.float64, device=self.device)
        t_mine = 0.0
        if T.n_states > 0 and T.n_items > 0:
            evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                   for _ in range(7)]
            for a, b in evs:
                a.record(self.torch_stream)
                rc = self.lib.sdp_sweep_partials(ctypes.byref(T.grid), ctypes.byref(T.c_tables),
                                                 self._ptr(J), self._ptr(T.part_val),
                                                 self._ptr(T.part_idx), self.stream)
                _cabi.check(rc, "sdp_sweep_partials")
                b.record(self.torch_stream)
            self.sync()
            t_mine = float(np.median([a.elapsed_time(b) for a, b in evs[2:]]))
        t = np.asarray(coll.all_gather_object(t_mine), dtype=float)
        if self.REBALANCE_SKEW is not None:      # test hook: pretend some slabs are slower
            t = t * np.asarray(self.REBALANCE_SKEW, dtype=float)[:len(t)]
        T.slab_times_ms = [float(x) for x in t]
        return rebalance_bounds(U_all, T.bounds, t, self.REBALANCE_TOLERANCE)

    # -- sweep tables -----------------------------------------------------
    # host cores for the per-state control_box scan of large grids (one rank; forked workers).
    # Opt-in (SDP_SCAN_PROCS=8): forking a process that holds a CUDA context and BLAS threads is
    # only safe for plain-numpy box functions; the scans above cover the common cases without it
    SCAN_PROCS = int(os.environ.get("SDP_SCAN_PROCS", "1"))
    SCAN_PARALLEL_MIN_STATES = 200 * 1000

    def _scan_boxes(self, solver, t_k, state_grid, n_grid, mode):
        """Pass 1 of a table build: the admissible box and control-grid sizes of every state of the
        grid.  Every rank scans an equal share (one vectorised call; else one call per distinct
        box; else per state, optionally on forked workers), the host table is replicated.
        Returns (HostStateTable of the whole grid, this rank's state tuples if they were made)."""
        sys = solver.sys
        coll = self.coll
        world, rank = coll.world, coll.rank
        nb_control = len(sys.control)
        eq = [n_grid * r // world for r in range(world + 1)]
        mine = None
        # the scan used to be by far the longest host stage: the last one is kept, so that a second
        # layout of the same problem (dense after factored, a re-cut of the slabs) does not repeat
        # it; DPSolver.clear_tables() drops it
        scan_key = (t_k, id(sys.control_box), repr(sorted(sys.params.items())) if sys.params else "",
                    tuple(float(c) for c in solver.control_steps),
                    tuple(g.tobytes() for g in state_grid), world)
        host_full = None
        if self._scan_cache is not None and self._scan_cache[0] == scan_key:
            host_full = self._scan_cache[1]
            # the box function may read globals / closure cells that changed since the scan
            # (the reference calls it afresh in every sweep): re-check three states
            probe = sorted({0, n_grid // 2, n_grid - 1})
            now = tb.scan_control_boxes(sys, solver.control_steps,
                                        [tb.state_tuples_at(state_grid, i, i + 1)[0] for i in probe], t_k)
            if not (np.array_equal(now.lo.view(np.int64), host_full.lo[probe].view(np.int64))
                    and np.array_equal(now.hi.view(np.int64), host_full.hi[probe].view(np.int64))
                    and np.array_equal(now.npts, host_full.npts[probe])):
                host_full = None
        if host_full is None:
            part = None
            if mode != "per_state":
                # one vectorised control_box call, trusted only if sample states agree
                # bit-for-bit with the reference's per-state calls
                part = tb.scan_control_boxes_batched(sys, solver.control_steps, state_grid,
                                                     eq[rank], eq[rank + 1], t_k)
            if part is None and mode != "per_state":
                # box functions that read only some of the state variables (the storage
                # examples): one call per distinct box, checked on sample states
                part = tb.scan_control_boxes_by_axes(sys, solver.control_steps, state_grid,
                                                     eq[rank], eq[rank + 1], t_k)
            if part is None and world == 1 and self.SCAN_PROCS > 1 and n_grid >= self.SCAN_PARALLEL_MIN_STATES:
                # box functions that do not vectorise (np.max((a, b)) on scalars, as in the
                # reference's examples): one call per state, on several host cores
                part = tb.scan_control_boxes_parallel(sys, solver.control_steps, state_grid,
                                                      eq[rank], eq[rank + 1], t_k, self.SCAN_PROCS)
            if part is None:
                mine = tb.state_tuples(state_grid, eq[rank], eq[rank + 1])
                part = tb.scan_control_boxes(sys, solver.control_steps, mine, t_k)
            parts = coll.all_gather_object((part.lo, part.hi, part.npts))
            host_full = tb.HostStateTable(n_grid, nb_control)
            host_full.lo = np.concatenate([p[0] for p in parts], axis=0)
            host_full.hi = np.concatenate([p[1] for p in parts], axis=0)
            host_full.npts = np.concatenate([p[2] for p in parts], axis=0)
            self._scan_cache = (scan_key, host_full)
        return host_full, mine

    def build_sweep_tables(self, solver, t_k=None, reuse=None):
        """Tabulate the user's callables over this rank's shard and build the tables on the
        device: `tablebuild.BuildPlan` (scan of the control boxes, cut over the ranks) and
        `tablebuild.ShardBuild` (layout, tabulation with its fall-backs, work list).  `reuse`: a
        SweepTables whose device buffers are recycled when the sizes match (time-dependent
        recursion).  With several ranks and slab_axis "auto" the grid is cut by columns when
        layout CF is expected to apply; if the built tables refuse it (same decision on every
        rank), the build starts again with slabs of rows."""
        try:
            return BuildPlan(self, solver, t_k).run(reuse)
        except _ColumnsNotApplicable:
            return BuildPlan(self, solver, t_k, forced_axis="rows").run(None)

    COLUMN_SEGS_PER_SM = int(os.environ.get("SDP_COLUMN_SEGS_PER_SM", "1"))
    # share of the tiles at the end of every (band, column) run whose work items are half as long
    COLUMN_TAIL_FRACTION = float(os.environ.get("SDP_COLUMN_TAIL_FRACTION", "0"))
    # launch shape of a band's sweep (SdpTables.col_launch_hint): 640 threads, round-robin - measured
    # on config #5 with ~10 column pieces per CTA (profiles/r2_emu_variants_bands.txt): 1.256 ms
    # against 1.346 ms for the 768-thread first-come-first-served shape that is best (1.146 against
    # 1.180 ms) when a CTA meets 3-4 long pieces
    BAND_LAUNCH_HINT = 640 | (1 << 16)

    def set_column_segments(self, T, n_ctas):
        """layout CF: re-cut the item list of built tables into `n_ctas` CTA segments
        (developer tuning, scripts/dev_column.py)"""
        assert T.column
        w = T.item_u_count_host[T.work_host]
        if T.item_order is not None:
            w = T.item_u_count_host[T.item_order.cpu().numpy()]
        seg = column_segments(w, n_ctas)
        T.seg_begin = self.to_device_packed([seg])[0]
        T.n_segs = len(seg) - 1
        T.c_tables = fill_c_tables(T)
        T.band_views = T.chunk_plan = None

    def _column_w_part_ok(self, T, W, n_cols, bands, valid, lam_w_plane):
        """layout CF: True when, in every column, the (x,w) part of all real states -
        partial cell index and weights of every perturbation node - is bit-identical to
        that of the column's first row (lane 0 of its first tile in the first band, the
        one the sweep kernels read)"""
        torch = _torch()
        live_all = torch.from_numpy(np.ascontiguousarray(valid)).to(self.device)
        planes = [T.cell_w] + [T.lam_w[j * lam_w_plane:(j + 1) * lam_w_plane].view(torch.int64)
                               for j in range(T.d - 1)]
        for t in planes:
            ref = None
            for tpc, t0, t1 in zip(bands["tiles"], bands["tile_begin"][:-1], bands["tile_begin"][1:]):
                v = t[t0 * W * 32:t1 * W * 32].view(n_cols, tpc, W, 32)
                if ref is None:
                    ref = v[:, :1, :, :1]
                live = live_all[t0 * 32:t1 * 32].view(n_cols, tpc, 1, 32)
                if not bool(((v == ref) | ~live).all().item()):
                    return False
        return True

    # layout CF on one rank, results for the host: the grid is swept in a few PIECES OF COLUMNS (see
    # _chunk_plan / sweep_to_host), each combined, mapped to control values and sent to its place
    # in the caller's arrays (2-D copies) while the next pieces are swept.  A piece of columns
    # costs a CTA no extra column table, unlike a band of ROWS, which costs every CTA a table load
    # and a drained barrier per (band, column) it meets: measured on config #5
    # (profiles/r1_column_tuning.txt, r2_emu_variants_bands.txt) the three row bands of round 1
    # took 1.256 ms per sweep against 1.146 ms for one band.  Row bands remain available
    # (SDP_COLUMN_BANDS = number of bands) and take the per-band path below.
    COLUMN_BANDS = os.environ.get("SDP_COLUMN_BANDS", "auto")    # "auto" (one band) | number of row bands
    # shares of the columns (by admissible controls) of the pieces, in sweep order: the copy of a
    # piece hides behind the pieces after it, the last piece's copy behind nothing
    COLUMN_PIECES = tuple(float(x) for x in os.environ.get("SDP_COLUMN_PIECES", "0.3,0.3,0.3,0.1").split(","))
    # ... with the cuts moved to multiples of the CTA count where that is close (column_piece_cuts)
    COLUMN_PIECES_ALIGN = os.environ.get("SDP_COLUMN_PIECES_ALIGN", "1") != "0"

    def _column_bands(self, row_weight, W):
        """row boundaries of the bands of layout CF for a slab whose rows weigh `row_weight`
        (admissible controls per row)"""
        n_rows = len(row_weight)
        mode = self.COLUMN_BANDS
        one = [0, n_rows]
        if self.coll.world > 1:
            return one               # the fused combine + exchange publishes one epoch per sweep
        if mode == "auto":
            return one               # results leave by pieces of columns (_column_piece_plan)
        k = max(1, int(mode))
        fractions = self.OVERLAP_FRACTIONS[:k - 1] + (1.0,) if k <= len(self.OVERLAP_FRACTIONS) \
            else tuple([1.0 / k] * k)
        if len(fractions) == 1 or n_rows < 64 * len(fractions):
            return one
        csum = np.cumsum(np.asarray(row_weight, dtype=np.float64))
        cuts, acc = [0], 0.0
        for f in fractions[:-1]:
            acc += f
            r = int(np.searchsorted(csum, acc * csum[-1], side="left")) + 1
            r = (r + 31) // 32 * 32                  # whole tiles: no padding lanes inside the slab
            if cuts[-1] < r < n_rows:
                cuts.append(r)
        return cuts + [n_rows]

    def _band_views(self, T):
        """layout CF: per band (SdpTables view for the combine pass, first state, states)"""
        if T.band_views is None:
            views = []
            B = T.bands
            for b, tpc in enumerate(B["tiles"]):
                v = _cabi.SdpTables.from_buffer_copy(T.c_tables)
                v.item_begin = T.c_tables.item_begin + 8 * int(B["tile_begin"][b])
                s0, s1 = int(B["rows"][b]) * T.n_cols, int(B["rows"][b + 1]) * T.n_cols
                v.n_states = s1 - s0
                v.tiles_per_col = int(tpc)
                if getattr(T, "pairs", False):
                    v.pos_row = T.pos_row.data_ptr() + 4 * 32 * int(sum(B["tiles"][:b]))
                views.append((v, s0, s1 - s0))
            T.band_views = views
        return T.band_views

    def _finalize(self, T, J_out, argmin, stream=None):
        """the combine pass: one launch, or for layout CF one per band"""
        stream = self.stream if stream is None else stream
        if not T.column:
            rc = self.lib.sdp_sweep_finalize(ctypes.byref(T.c_tables), self._ptr(T.part_val),
                                             self._ptr(T.part_idx), self._ptr(J_out), self._ptr(argmin), stream)
            _cabi.check(rc, "sdp_sweep_finalize")
            return
        for v, s0, ns in self._band_views(T):
            rc = self.lib.sdp_sweep_finalize(ctypes.byref(v), self._ptr(T.part_val), self._ptr(T.part_idx),
                                             ctypes.c_void_p(J_out.data_ptr() + 8 * s0),
                                             ctypes.c_void_p(argmin.data_ptr() + 4 * s0), stream)
            _cabi.check(rc, "sdp_sweep_finalize")

    def sweep_local(self, T, J_prev, events=None, J_out=None):
        """Enqueue K1 on this rank's slab.  J_prev: device fp64 [n_grid].
        Results land in `J_out` (default T.J_out) / T.argmin (slab-local).  `events`: optional
        (start, end) torch.cuda.Event pair recorded around the streaming kernel
        alone (bench roofline)."""
        J_out = T.J_out if J_out is None else J_out
        if events is None and not T.column:
            rc = self.lib.sdp_sweep(ctypes.byref(T.grid), ctypes.byref(T.c_tables), self._ptr(J_prev),
                                    self._ptr(T.part_val), self._ptr(T.part_idx),
                                    self._ptr(J_out), self._ptr(T.argmin), self.stream)
            _cabi.check(rc, "sdp_sweep")
            return
        if events is not None:
            events[0].record(self.torch_stream)
        rc = self.lib.sdp_sweep_partials(ctypes.byref(T.grid), ctypes.byref(T.c_tables),
                                         self._ptr(J_prev), self._ptr(T.part_val),
                                         self._ptr(T.part_idx), self.stream)
        _cabi.check(rc, "sdp_sweep_partials")
        if events is not None:
            events[1].record(self.torch_stream)
        self._finalize(T, J_out, T.argmin)

    # Device-resident iterations (solve_value_iteration, the bench loop) may leave the flag wait
    # of a sweep's exchange to the NEXT sweep, whose first kernel then starts with it
    # (sdp_sweep_partials_after): one launch less per sweep.  Every other consumer of J calls
    # flush_exchange() first.  SDP_FOLD_WAIT=0 keeps the separate sdp_p2p_wait launch.
    FOLD_WAIT = os.environ.get("SDP_FOLD_WAIT", "1") != "0"
    _pending_wait = None

    def flush_exchange(self):
        """enqueue the flag wait a sweep(..., defer_wait=True) left pending"""
        pend, self._pending_wait = self._pending_wait, None
        if pend is not None:
            rc = self.lib.sdp_p2p_wait(ctypes.byref(pend), self.stream)
            _cabi.check(rc, "sdp_p2p_wait")

    def sweep(self, T, J_prev, J_new, rel_ref_index=None, ref_out=None, resid_out=None,
              events=None, defer_wait=False, want_argmin=True):
        """One full Bellman sweep: K1 on the slab, all-gather of the J slab into
        J_new (device fp64 [n_grid]), optional relative-DP shift and optional
        sup-norm residual max|J_new - J_prev| (all-reduced).
        `defer_wait`: the caller's next use of J_new is another sweep (or it calls
        flush_exchange() itself): the arrival of the peers' slabs is then awaited by that
        sweep's first kernel.
        `want_argmin` False: an intermediate sweep of a device-resident loop, whose policy
        nobody reads - the combine kernel then sends J alone to the peers (the shard's own
        argmin is still written; gather_argmin falls back to collecting those)."""
        n = T.n_states
        sb = T.state_begin
        px = self._peer.get(J_new.numel()) if self.coll.world > 1 else None
        k_new = px.index_of(J_new) if px is not None else None
        pend, self._pending_wait = self._pending_wait, None
        if k_new is None and pend is not None:
            self._pending_wait = pend
            self.flush_exchange()
            pend = None
        if k_new is not None:
            # fused combine + all-gather: K1, then the combine kernel stores the slab
            # into every rank's J_new over NVLink and publishes the epoch
            if events is not None:
                events[0].record(self.torch_stream)
            if pend is not None:
                rc = self.lib.sdp_sweep_partials_after(ctypes.byref(T.grid), ctypes.byref(T.c_tables),
                                                       self._ptr(J_prev), self._ptr(T.part_val),
                                                       self._ptr(T.part_idx), ctypes.byref(pend), self.stream)
                _cabi.check(rc, "sdp_sweep_partials_after")
            else:
                rc = self.lib.sdp_sweep_partials(ctypes.byref(T.grid), ctypes.byref(T.c_tables),
                                                 self._ptr(J_prev), self._ptr(T.part_val),
                                                 self._ptr(T.part_idx), self.stream)
                _cabi.check(rc, "sdp_sweep_partials")
            if events is not None:
                events[1].record(self.torch_stream)
            P_out = px.peers[k_new] if want_argmin else px.peers_J_only[k_new]
            if T.col_bounds is not None:
                rc = self.lib.sdp_sweep_finalize_p2p_cols(
                    ctypes.byref(T.c_tables), self._ptr(T.part_val), self._ptr(T.part_idx), self._ptr(T.argmin),
                    ctypes.byref(P_out), T.col_bounds[-1], T.col_bounds[self.coll.rank], self.stream)
                _cabi.check(rc, "sdp_sweep_finalize_p2p_cols")
            else:
                rc = self.lib.sdp_sweep_finalize_p2p(ctypes.byref(T.c_tables), self._ptr(T.part_val),
                                                     self._ptr(T.part_idx), self._ptr(T.argmin),
                                                     ctypes.byref(P_out), sb, self.stream)
                _cabi.check(rc, "sdp_sweep_finalize_p2p")
            self._argmin_in_px = bool(want_argmin)
            if defer_wait and self.FOLD_WAIT and rel_ref_index is None and resid_out is None:
                self._pending_wait = px.peers[k_new]
            else:
                rc = self.lib.sdp_p2p_wait(ctypes.byref(px.peers[k_new]), self.stream)
                _cabi.check(rc, "sdp_p2p_wait")
        else:
            self._argmin_in_px = False
            if self.coll.world == 1:
                self.sweep_local(T, J_prev, events, J_out=J_new)     # (one rank: straight into J_new)
            else:
                self.sweep_local(T, J_prev, events)
            if self.coll.world == 1:
                pass
            elif T.col_bounds is not None:
                self.coll.all_gather_indexed(T.J_out[:n], T.gather_maxc, T.gather_index, out=J_new)
            else:
                self.coll.all_gather_slabs(T.J_out[:n], T.bounds, out=J_new)
        if rel_ref_index is not None:
            rc = self.lib.sdp_rel_shift(self._ptr(J_new), J_new.numel(), int(rel_ref_index),
                                        self._ptr(ref_out), self.stream)
            _cabi.check(rc, "sdp_rel_shift")
        if resid_out is not None:
            if T.col_bounds is not None:
                # every rank holds all of J: any partition of the grid does for the residual
                world, rank, n_grid = self.coll.world, self.coll.rank, J_new.numel()
                sb = n_grid * rank // world
                n = n_grid * (rank + 1) // world - sb
            a = J_new[sb:sb + n]
            b = J_prev[sb:sb + n]
            rc = self.lib.sdp_supnorm_diff(self._ptr(a), self._ptr(b), n, self._ptr(resid_out),
                                           self.stream)
            _cabi.check(rc, "sdp_supnorm_diff")
            self.coll.all_reduce_max(resid_out)

    # -- one sweep with host results, D2H overlapped with compute -------------
    OVERLAP_MIN_BACKUPS = 100 * 1000 * 1000     # below this the result copy is not worth hiding
    OVERLAP_MIN_ITEMS = 4096
    OVERLAP_FRACTIONS = (0.45, 0.25, 0.15, 0.10, 0.05)

    def can_overlap_results(self, T):
        if T.column and len(T.bands["tiles"]) < 2 and (T.n_cols < 2 or T.col_bounds is not None):
            return False             # layout CF streams its results by pieces of columns (or row bands)
        return (self._cuda and self.coll.world == 1 and T.n_items >= self.OVERLAP_MIN_ITEMS
                and T.n_backups_local >= self.OVERLAP_MIN_BACKUPS
                and os.environ.get("SDP_OVERLAP", "1") != "0")

    def _chunk_plan(self, T):
        """cut the slab's work units (states, or tiles of 32 states) into a few runs of
        decreasing size; each run is swept by its own launches (sub-range views of the
        same tables: shifted item / item_begin pointers), so that its results can
        travel to the host while the next run computes"""
        if T.chunk_plan is not None:
            return T.chunk_plan
        if T.column and len(T.bands["tiles"]) == 1:
            T.chunk_plan = self._column_piece_plan(T)
            return T.chunk_plan
        if T.column:
            # one run per band: its own CTA segments over the band's items (absolute item
            # indices, the column tables are tabulated once before the first run)
            plan = []
            tb0 = T.bands["tile_begin"]
            for b, (view, s0, ns) in enumerate(self._band_views(T)):
                # (positions of the work list - every item, or with two rows per lane the items
                # of the first tile of every pair - that belong to the band)
                i0, i1 = (int(np.searchsorted(T.work_host, T.item_begin_host[tb0[k]])) for k in (b, b + 1))
                seg = i0 + column_segments(T.item_u_count_host[T.work_host[i0:i1]],
                                           T.sm_count * self.COLUMN_SEGS_PER_SM)
                seg_dev = self.to_device_packed([seg])[0]
                cp = _cabi.SdpTables.from_buffer_copy(T.c_tables)
                cp.seg_begin, cp.n_segs, cp.col_table_ready = seg_dev.data_ptr(), len(seg) - 1, 1
                # a band is walked in the list's own order: many short column pieces per CTA
                cp.item_order = T.work_dev.data_ptr() if T.work_dev is not None else 0
                cp.run_end = T.run_end.data_ptr()
                cp.col_launch_hint = self.BAND_LAUNCH_HINT
                plan.append(dict(tab_p=cp, tab_f=view, s0=s0, s1=s0 + ns, keep=seg_dev,
                                 pv=ctypes.c_void_p(T.part_val.data_ptr()),
                                 pi=ctypes.c_void_p(T.part_idx.data_ptr())))
            T.chunk_plan = plan
            return plan
        us = 32 if T.tiled else 1
        n_units = len(T.unit_U_host)
        csum = np.cumsum(T.unit_U_host)
        total = float(csum[-1])
        cuts = [0]
        acc = 0.0
        for f in self.OVERLAP_FRACTIONS[:-1]:
            acc += f
            b = int(np.searchsorted(csum, acc * total, side="left")) + 1
            cuts.append(min(max(b, cuts[-1]), n_units))
        cuts.append(n_units)
        plan = []
        width = 32 if T.tiled else 1
        for a, b in zip(cuts[:-1], cuts[1:]):
            if b <= a:
                continue
            i0, i1 = int(T.item_begin_host[a]), int(T.item_begin_host[b])
            s0, s1 = a * us, min(b * us, T.n_states)
            cp = _cabi.SdpTables.from_buffer_copy(T.c_tables)
            cp.items = T.c_tables.items + _cabi.ITEM_DTYPE.itemsize * i0
            cp.n_items = i1 - i0
            cf = _cabi.SdpTables.from_buffer_copy(T.c_tables)
            cf.item_begin = T.c_tables.item_begin + 8 * a
            cf.n_states = s1 - s0
            plan.append(dict(tab_p=cp, tab_f=cf, s0=s0, s1=s1,
                             pv=ctypes.c_void_p(T.part_val.data_ptr() + 8 * width * i0),
                             pi=ctypes.c_void_p(T.part_idx.data_ptr() + 4 * width * i0)))
        T.chunk_plan = plan
        return plan

    def _column_piece_plan(self, T):
        """layout CF, one band: the columns cut into a few pieces of decreasing weight
        (COLUMN_PIECES).  The items of a column are consecutive, so a piece is a range of the
        work list with its own CTA segments (absolute positions; the column tables are tabulated
        once before the first piece) and a view of the tables on its columns for the combine."""
        tpc = int(T.bands["tiles"][0])
        n_cols = T.n_cols
        n_rows = T.n_states // n_cols
        first_item = T.item_begin_host[np.arange(n_cols + 1, dtype=np.int64) * tpc]      # per column
        csum = np.concatenate([[0], np.cumsum(T.item_u_count_host, dtype=np.float64)])[first_item]
        cuts = column_piece_cuts(csum, self.COLUMN_PIECES,
                                 T.sm_count * self.COLUMN_SEGS_PER_SM if self.COLUMN_PIECES_ALIGN else 0)
        plan = []
        for c0, c1 in zip(cuts[:-1], cuts[1:]):
            # (positions of the work list - every item, or with two rows per lane the items of the
            # first tile of every pair - that belong to the piece)
            i0, i1 = (int(np.searchsorted(T.work_host, first_item[c])) for c in (c0, c1))
            seg = i0 + column_segments(T.item_u_count_host[T.work_host[i0:i1]],
                                       T.sm_count * self.COLUMN_SEGS_PER_SM)
            seg_dev = self.to_device_packed([seg])[0]
            cp = _cabi.SdpTables.from_buffer_copy(T.c_tables)
            cp.seg_begin, cp.n_segs, cp.col_table_ready = seg_dev.data_ptr(), len(seg) - 1, 1
            cp.item_order = T.work_dev.data_ptr() if T.work_dev is not None else 0
            cp.run_end = T.run_end.data_ptr()
            view = _cabi.SdpTables.from_buffer_copy(T.c_tables)
            view.item_begin = T.c_tables.item_begin + 8 * c0 * tpc
            view.n_cols = c1 - c0
            view.n_states = n_rows * (c1 - c0)
            plan.append(dict(kind="cols", tab_p=cp, tab_f=view, c0=c0, c1=c1, n_rows=n_rows, keep=seg_dev,
                             pv=ctypes.c_void_p(T.part_val.data_ptr()),
                             pi=ctypes.c_void_p(T.part_idx.data_ptr())))
        return plan

    def _columns_to_host(self, T, ch, J_new, pol, J_pin, pol_pin):
        """on the copy stream: the columns [c0, c1) of J and of the policy (device, grid order) into
        the same columns of the C-order host arrays - one 2-D copy each"""
        nc, n_cols, c0, c1, n_rows = T.nb_control, T.n_cols, ch["c0"], ch["c1"], ch["n_rows"]
        cs = ctypes.c_void_p(self._copy.cuda_stream)
        rc = self.lib.sdp_memcpy_2d(ctypes.c_void_p(J_pin.data_ptr() + 8 * c0), 8 * n_cols,
                                    ctypes.c_void_p(J_new.data_ptr() + 8 * c0), 8 * n_cols,
                                    8 * (c1 - c0), n_rows, cs)
        _cabi.check(rc, "sdp_memcpy_2d")
        if nc:
            rc = self.lib.sdp_memcpy_2d(ctypes.c_void_p(pol_pin.data_ptr() + 8 * nc * c0), 8 * nc * n_cols,
                                        ctypes.c_void_p(pol.data_ptr() + 8 * nc * c0), 8 * nc * n_cols,
                                        8 * nc * (c1 - c0), n_rows, cs)
            _cabi.check(rc, "sdp_memcpy_2d")

    def sweep_to_host(self, T, J_prev, J_new, while_waiting=None):
        """One sweep of a single-rank slab, returning (J, pol) as host arrays in
        page-locked memory.  The slab is swept in a few runs (`_chunk_plan`: ranges of
        states, row bands of layout CF, or - layout CF with one band, the default - pieces
        of columns) on two alternating streams (so that the tail of one run is filled by
        the next); as soon as a run is combined and its argmin mapped to control values
        (K3; one launch does both for a piece of columns), a copy stream sends that run's
        J and policy to their place in the host arrays while the following runs still
        compute.  Same kernels on sub-ranges of the same tables: bit-identical to `sweep`.
        (stodynprog.py:496-499,517-521: J_k and pol_k are C-order arrays over the grid.)"""
        torch = _torch()
        dev = self.device
        n, nc = T.n_states, T.nb_control
        if not hasattr(self, "_side"):
            self._side = [torch.cuda.Stream(dev), torch.cuda.Stream(dev)]
            self._copy = torch.cuda.Stream(dev)
        main = torch.cuda.current_stream(dev)
        # developer timeline (scripts/dev_e2e_timeline.py): a list that receives (label, event)
        trace = getattr(self, "_trace", None)

        def mark(label, stream):
            if trace is not None:
                e = torch.cuda.Event(enable_timing=True)
                e.record(stream)
                trace.append((label, e))
        mark("J on the device", main)
        pol = torch.empty((n, nc), dtype=torch.float64, device=dev)
        J_pin = self.host_result_buffer((n,), torch.float64)
        pol_pin = self.host_result_buffer((n, nc), torch.float64)
        if T.column:
            rc = self.lib.sdp_column_table(ctypes.byref(T.grid), ctypes.byref(T.c_tables), self._ptr(J_prev),
                                           self.stream)
            _cabi.check(rc, "sdp_column_table")
        ev0 = torch.cuda.Event()
        ev0.record(main)
        mark("column tables", main)
        plan = self._chunk_plan(T)
        after = None
        for k, ch in enumerate(plan):
            st = self._side[k % 2]
            sp = ctypes.c_void_p(st.cuda_stream)
            st.wait_event(ev0)
            if after is not None:
                st.wait_event(after)       # (the last piece of columns starts after the combine before it)
                after = None
            rc = self.lib.sdp_sweep_partials(ctypes.byref(T.grid), ctypes.byref(ch["tab_p"]),
                                             self._ptr(J_prev), ch["pv"], ch["pi"], sp)
            _cabi.check(rc, "sdp_sweep_partials")
            mark("run %d swept" % k, st)
            if ch.get("kind") == "cols":
                # the combine of a piece runs beside the sweep of the next one (small CTAs that fit
                # next to the resident streaming CTAs; it takes ~180 us that way, hidden) - except the
                # last two: the results of the last-but-one piece would leave too late, so its
                # combine (15 us on the free GPU) goes BEFORE the last sweep, and nothing runs
                # beside the last combine
                beside = k + 2 < len(plan)
                ev = torch.cuda.Event()
                rc = self.lib.sdp_sweep_finalize_cols(
                    ctypes.byref(ch["tab_f"]), self._ptr(T.part_val), self._ptr(T.part_idx), self._ptr(J_new),
                    self._ptr(T.argmin), T.n_cols, ch["c0"], nc, self._ptr(T.lo_dev), self._ptr(T.hi_dev),
                    self._ptr(T.npts_dev), self._ptr(pol) if nc else ctypes.c_void_p(0), int(beside), sp)
                _cabi.check(rc, "sdp_sweep_finalize_cols")
                ev.record(st)
                if k + 2 == len(plan):
                    after = ev
                mark("run %d combined + mapped" % k, st)
                self._copy.wait_event(ev)
                self._columns_to_host(T, ch, J_new, pol, J_pin, pol_pin)
                mark("run %d on the host" % k, self._copy)
                continue
            s0, s1 = ch["s0"], ch["s1"]
            rc = self.lib.sdp_sweep_finalize(ctypes.byref(ch["tab_f"]), self._ptr(T.part_val),
                                             self._ptr(T.part_idx),
                                             ctypes.c_void_p(J_new.data_ptr() + 8 * s0),
                                             ctypes.c_void_p(T.argmin.data_ptr() + 4 * s0), sp)
            _cabi.check(rc, "sdp_sweep_finalize")
            if nc:
                rc = self.lib.sdp_policy_values(
                    s1 - s0, nc, ctypes.c_void_p(T.lo_dev.data_ptr() + 8 * nc * s0),
                    ctypes.c_void_p(T.hi_dev.data_ptr() + 8 * nc * s0),
                    ctypes.c_void_p(T.npts_dev.data_ptr() + 4 * nc * s0),
                    ctypes.c_void_p(T.argmin.data_ptr() + 4 * s0),
                    ctypes.c_void_p(pol.data_ptr() + 8 * nc * s0), sp)
                _cabi.check(rc, "sdp_policy_values")
            ev = torch.cuda.Event()
            ev.record(st)
            mark("run %d combined + mapped" % k, st)
            self._copy.wait_event(ev)
            with torch.cuda.stream(self._copy):
                J_pin[s0:s1].copy_(J_new[s0:s1], non_blocking=True)
                if nc:
                    pol_pin[s0:s1].copy_(pol[s0:s1], non_blocking=True)
            mark("run %d on the host" % k, self._copy)
        done = torch.cuda.Event()
        done.record(self._copy)
        main.wait_event(done)
        if while_waiting is not None:
            while_waiting()          # host work hidden behind the sweep (the GPU is busy)
        out = self.result_array(J_pin), self.result_array(pol_pin)      # (wrapped while the GPU works)
        done.synchronize()
        return out

    def gather_argmin(self, T):
        """full-grid int32 argmin (device) of the last sweep.  With the peer-memory exchange every
        rank already holds it (the combine kernel stores the argmin next to J, SdpPeers.A): valid
        until the next sweep; otherwise gathered over the ranks"""
        if self.coll.world > 1 and T.host_full is not None:
            px = self._peer.get(int(T.host_full.lo.shape[0]))
            if px is not None and getattr(self, "_argmin_in_px", False):
                self.flush_exchange()
                return px.argmin
        if T.col_bounds is not None:
            return self.coll.all_gather_indexed(T.argmin[:T.n_states], T.gather_maxc, T.gather_index)
        return self.coll.all_gather_slabs(T.argmin[:T.n_states], T.bounds)

    def policy_values(self, T, argmin_full):
        """K3: full-grid argmin (device int32 [N]) -> control values (device fp64 [N][nc])"""
        torch = _torch()
        n = argmin_full.numel()
        nc = T.nb_control
        pol = torch.empty((n, nc), dtype=torch.float64, device=self.device)
        if nc:
            rc = self.lib.sdp_policy_values(n, nc, self._ptr(T.lo_dev), self._ptr(T.hi_dev),
                                            self._ptr(T.npts_dev), self._ptr(argmin_full),
                                            self._ptr(pol), self.stream)
            _cabi.check(rc, "sdp_policy_values")
        return pol

    # Result arrays are handed to the caller as numpy views of page-locked buffers (no
    # extra host copy, and the next call can DMA them back without staging).  Page-locked
    # memory is a limited resource and a caller may keep every J_k of a long iteration:
    # above this budget of LIVE result bytes new results go to ordinary pageable memory.
    PINNED_RESULT_BUDGET = int(os.environ.get("SDP_PINNED_RESULT_BUDGET", str(4 << 30)))
    _pinned_live = [0]

    def host_result_buffer(self, shape, dtype):
        """uninitialised host tensor for a result: page-locked while the budget lasts"""
        torch = _torch()
        nbytes = int(np.prod(shape)) * torch.empty(0, dtype=dtype).element_size()
        if not self._cuda or Engine._pinned_live[0] + nbytes > self.PINNED_RESULT_BUDGET:
            return torch.empty(shape, dtype=dtype)
        return torch.empty(shape, dtype=dtype, pin_memory=True)

    def result_array(self, t):
        """numpy view of a host result tensor; a page-locked one is counted against the
        budget until the caller drops the array (views made from it keep it alive)"""
        import weakref
        a = t.numpy()
        if self._cuda and t.is_pinned():
            nbytes = a.nbytes
            live = Engine._pinned_live
            live[0] += nbytes

            def release(n=nbytes, live=live):
                live[0] -= n
            weakref.finalize(a, release)
        return a

    def to_host(self, *tensors, while_waiting=None):
        """device tensors -> fresh numpy arrays (through pinned buffers, one sync);
        `while_waiting()` runs on the host between the enqueue and the synchronisation"""
        torch = _torch()
        self.flush_exchange()
        if not self._cuda:
            if while_waiting is not None:
                while_waiting()
            return [t.numpy().copy() for t in tensors]
        outs = [self.host_result_buffer(tuple(t.shape), t.dtype) for t in tensors]
        for o, t in zip(outs, tensors):
            o.copy_(t, non_blocking=True)
        if while_waiting is not None:
            while_waiting()
        torch.cuda.current_stream(self.device).synchronize()
        return [self.result_array(o) for o in outs]

    def _pinned_scratch(self, n_doubles):
        """page-locked fp64 scratch of at least `n_doubles`, kept on the engine (allocating and
        pinning 100+ MB costs as much as copying it); None without CUDA"""
        if not self._cuda:
            return None
        torch = _torch()
        buf = getattr(self, "_pin_scratch", None)
        if buf is None or buf.numel() < n_doubles:
            self._pin_scratch = None
            buf = self._pin_scratch = torch.empty(n_doubles, dtype=torch.float64, pin_memory=True)
        return buf

    # -- time-dependent recursion, fast path ----------------------------------
    RECURSION_MAX_G_BYTES = 8 << 30      # per-instant stage-cost tables kept resident

    def recursion_fast(self, solver, t_ini, t_fin, J_fin, J_out, pol_out):
        """bellman_recursion (stodynprog.py:536-591) for systems whose dynamics and admissible
        controls do not depend on the instant, only the stage cost does - the reference's
        time-dependent examples (examples/01 .../pv_storage_control.py:43-65: the PV production
        enters the cost alone).  The cell / weight tables are then the same at every instant:
        they are built once, the cost is tabulated for all instants up front, the T sweeps
        are enqueued back to back with J and the policy staying on the device, and one copy
        brings (J, pol) of all instants to the host.

        Nothing is assumed: the box scan and the batched dyn evaluation of the first, middle
        and last instant are compared bit for bit, and at every instant dyn / control_box of
        one sample state (another one each time) are compared with the tables and the batched
        cost is checked on sample states against the reference's per-state call.  Any
        difference -> returns None and the caller takes the per-instant path.
        Returns a dict of timings on success."""
        import time
        torch = _torch()
        t0 = time.perf_counter()
        sys = solver.sys
        if self.coll.world > 1 or t_fin - t_ini < 3:
            return None
        t_base = t_fin - 1
        solver._keep_staging = True
        try:
            T = self.build_sweep_tables(solver, t_base)
        finally:
            solver._keep_staging = False
        rec = getattr(T, "build_record", None)
        if rec is None or T.n_states != len(rec["desc"]):
            return None
        d, nc, W = T.d, T.nb_control, T.W
        host, cols, outs0 = rec["host"], rec["cols"], rec["outs"]
        S = T.n_states
        g0 = outs0[-1]
        n_T = t_fin - t_ini
        g_len = T.g.numel()
        if n_T * g_len * 8 > self.RECURSION_MAX_G_BYTES:
            return None
        state_grid = [np.asarray(g, dtype=float) for g in solver.state_grid]
        w_args, w_shape, _ = tb.perturb_layout(rec["w_grid"])
        state_of = lambda i: tuple(c[i] for c in cols)            # noqa: E731

        def same_bits(a, b):
            return a.shape == b.shape and np.array_equal(a.view(np.int64), b.view(np.int64))

        # 1. dyn / control_box at the first and the middle instant against the last one
        for t_chk in sorted({t_ini, (t_ini + t_fin) // 2}):
            if t_chk == t_base:
                continue
            box = tb.scan_control_boxes(sys, solver.control_steps, [state_of(i) for i in range(S)], t_chk)
            if not (same_bits(box.lo, host.lo) and same_bits(box.hi, host.hi) and np.array_equal(box.npts, host.npts)):
                return None
            dyn_t, _ = tb._eval_state_chunk(sys, cols, host.lo, host.hi, host.npts, w_args, t_chk, W,
                                            self._grid_cache, w_shape, only="dyn")
            if not all(same_bits(a, b) for a, b in zip(dyn_t, outs0[:d])):
                return None

        # 2. the stage cost of every instant (one batched call each), checked on sample states
        # (filled in place in page-locked memory kept between recursions: one asynchronous upload)
        g_pin = self._pinned_scratch(n_T * g0.size)
        g_src = (g_pin.numpy() if g_pin is not None else np.empty(n_T * g0.size)).reshape((n_T,) + g0.shape)
        k_base = t_base - t_ini
        g_src[k_base] = g0
        for k in range(n_T):
            t_k = t_ini + k
            if t_k == t_base:
                continue
            i_chk = (7 * k) % S
            x_chk = state_of(i_chk)
            box = tb.scan_control_boxes(sys, solver.control_steps, [x_chk], t_k)
            if not (same_bits(box.lo[0], host.lo[i_chk]) and same_bits(box.hi[0], host.hi[i_chk])
                    and np.array_equal(box.npts[0], host.npts[i_chk])):
                return None
            (g_t,), nmax = tb._eval_state_chunk(sys, cols, host.lo, host.hi, host.npts, w_args, t_k, W,
                                                self._grid_cache, w_shape, only="cost")
            if g_t.shape != g0.shape:
                return None
            full = tuple(int(n) for n in host.npts[i_chk]) + (W,)
            for i_s, what in ((i_chk, None), ((i_chk + S // 2) % S, "cost")):
                compact, cdims, U = tb._eval_one_state(sys, state_of(i_s), host, i_s, w_args, t_k, W, w_shape,
                                                       only=what)
                cdims = tuple(cdims)
                pairs = [(g_t, compact[-1])] if what == "cost" else \
                    list(zip(list(outs0[:d]) + [g_t], compact))
                for a, (ref, u_eff, w_eff) in pairs:
                    row = a[i_s if a.shape[0] > 1 else 0]
                    sl = tuple(slice(0, cdims[c] if row.shape[c] > 1 else 1) for c in range(nc))
                    shape = (cdims if u_eff > 1 else (1,) * nc) + (w_eff,)
                    fullb = cdims + (W,)
                    got = np.ascontiguousarray(np.broadcast_to(row[sl], fullb))
                    want = np.ascontiguousarray(np.broadcast_to(ref.reshape(shape), fullb))
                    if not same_bits(got, want):
                        return None
            g_src[k] = g_t
        t_tab = time.perf_counter()

        # 3. device: staging of instant t_base + the cost of all instants behind it; per-instant
        # descriptors differ only in where the cost is read
        n_stag = rec["n_staging"]
        g_size = g0.size
        stag_all = torch.empty(n_stag + n_T * g_size, dtype=torch.float64, device=self.device)
        stag_all[:n_stag].copy_(rec["stag_dev"])
        if g_pin is not None:
            stag_all[n_stag:].copy_(g_pin[:n_T * g_size], non_blocking=True)
        else:
            stag_all[n_stag:].copy_(self.to_device(g_src.reshape(-1)))
        desc_all = np.repeat(rec["desc"][None, :], n_T, axis=0)
        shift = n_stag + np.arange(n_T, dtype=np.int64) * g_size - rec["g_base"]
        desc_all["src"][:, :, d] += shift[:, None]
        desc_dev = self.to_device_packed([desc_all.reshape(-1)])[0]
        desc_bytes = desc_all.dtype.itemsize * S
        g_all = torch.empty((n_T, g_len), dtype=torch.float64, device=self.device)
        for k in range(n_T):
            rec["launch"](ctypes.c_void_p(desc_dev.data_ptr() + k * desc_bytes), self._ptr(stag_all),
                          ctypes.c_void_p(g_all.data_ptr() + 8 * k * g_len))

        # 4. the T sweeps back to back, J and the policy on the device
        n_grid = S
        J_all = torch.empty((n_T + 1, n_grid), dtype=torch.float64, device=self.device)
        J_all[n_T].copy_(self.to_device(np.ascontiguousarray(np.asarray(J_fin, dtype=np.float64).reshape(-1))))
        arg_all = torch.empty((n_T, n_grid), dtype=torch.int32, device=self.device)
        pol_all = torch.empty((n_T, n_grid, max(nc, 1)), dtype=torch.float64, device=self.device)
        self.sync()
        t_up = time.perf_counter()
        for k in range(n_T - 1, -1, -1):
            v = _cabi.SdpTables.from_buffer_copy(T.c_tables)
            v.g = g_all.data_ptr() + 8 * k * g_len
            rc = self.lib.sdp_sweep(ctypes.byref(T.grid), ctypes.byref(v), self._ptr(J_all[k + 1]),
                                    self._ptr(T.part_val), self._ptr(T.part_idx), self._ptr(J_all[k]),
                                    self._ptr(arg_all[k]), self.stream)
            _cabi.check(rc, "sdp_sweep")
            if nc:
                rc = self.lib.sdp_policy_values(n_grid, nc, self._ptr(T.lo_dev), self._ptr(T.hi_dev),
                                                self._ptr(T.npts_dev), self._ptr(arg_all[k]),
                                                self._ptr(pol_all[k]), self.stream)
                _cabi.check(rc, "sdp_policy_values")
        J_h, pol_h = self.to_host(J_all[:n_T], pol_all)
        t_end = time.perf_counter()
        J_out[...] = J_h.reshape(J_out.shape)
        if nc:
            pol_out[...] = pol_h.reshape(pol_out.shape)
        return {"tabulate_s": t_tab - t0, "upload_build_s": t_up - t_tab, "sweeps_s": t_end - t_up,
                "instants": n_T, "tables": T}

    # -- policy tables ----------------------------------------------------
    def build_policy_tables(self, solver, pol, t_k=None, deterministic=False):
        """Evaluate dyn/cost for the fixed policy on the whole grid exactly as
        eval_policy does (one broadcast call, stodynprog.py:731-755), expand on the
        host to dense [d][W][N] coordinates and run the cell search (K0a) for this
        rank's equal-count slab.

        t_k: the instant, passed first to dyn/cost (as bellman_recursion does).
        deterministic: accept a system without perturbation (W = 1, p = [1]); eval_policy
        leaves it False and raises IndexError there, like the reference (:726)."""
        torch = _torch()
        sys = solver.sys
        state_grid_1d = [np.asarray(g, dtype=float) for g in solver.state_grid]
        state_dims = tuple(len(g) for g in state_grid_1d)
        nb_state = len(state_dims)
        nb_control = len(sys.control)
        grid = _cabi.make_grid(state_grid_1d)
        n_grid = int(np.prod(state_dims))
        if not deterministic:
            solver.perturb_grid[0]                    # IndexError if deterministic, like :726
        w_args, w_shape, W = tb.perturb_layout(solver.perturb_grid)
        w_proba = tb.joint_proba(solver.perturb_proba)
        n_w_axes = len(w_shape)
        state_grid = tuple(np.reshape(g, (1,) * i + (-1,) + (1,) * (nb_state - 1 - i + n_w_axes))
                           for i, g in enumerate(solver.state_grid))
        u_k = [pol[..., i].reshape(state_dims + (1,) * n_w_axes) for i in range(nb_control)]
        args = ((t_k,) if t_k is not None else ()) + state_grid + tuple(u_k) + w_args
        x_next = sys.dyn(*args, **sys.params)
        g_k = sys.cost(*args, **sys.params)
        if n_w_axes == 0:
            # no perturbation: outputs broadcast to the state grid; one node of probability 1
            x_next = tuple(self._as_full(c, state_dims)[..., None] for c in x_next)
            g_k = self._as_full(g_k, state_dims)[..., None]
        elif n_w_axes > 1:
            # one trailing axis: the C-order flattened product of the perturbation axes
            x_next = tuple(tb._fold_w(self._as_full(c, state_dims + w_shape), nb_state, w_shape, "dyn")
                           for c in x_next)
            g_k = tb._fold_w(self._as_full(g_k, state_dims + w_shape), nb_state, w_shape, "cost")
        full = state_dims + (W,)
        world, rank = self.coll.world, self.coll.rank
        bounds = [n_grid * r // world for r in range(world + 1)]
        sb, se = bounds[rank], bounds[rank + 1]
        n = se - sb

        def dense_wn(a, allow_compact_w):
            a = np.asarray(a)
            if a.dtype != np.float64:
                a = a.astype(float)
            if a.ndim > len(full):
                raise ValueError("dyn/cost output of rank %d does not broadcast to %s" % (a.ndim, full))
            a = a.reshape((1,) * (len(full) - a.ndim) + a.shape)
            if allow_compact_w and a.shape[-1] == 1:
                flat = np.broadcast_to(a, state_dims + (1,)).reshape(n_grid)
                return np.ascontiguousarray(flat[sb:se]), 0
            flat = np.broadcast_to(a, full).reshape(n_grid, W)
            return np.ascontiguousarray(flat[sb:se].T), 1     # [W][n]

        P = PolicyTables()
        P.grid, P.W, P.bounds, P.state_begin, P.n_states = grid, W, bounds, sb, n
        coords = np.stack([dense_wn(c, False)[0].reshape(-1) for c in x_next]) if n else \
            np.zeros((nb_state, 0))
        g_arr, g_per_w = dense_wn(g_k, True)
        P.g_per_w = g_per_w
        P.lam_plane = W * n
        s_dev = self.to_device(coords)
        P.cell = torch.empty(max(W * n, 1), dtype=torch.int32, device=self.device)
        P.lam = torch.empty(max(W * n, 1) * nb_state, dtype=torch.float64, device=self.device)
        rc = self.lib.sdp_cell_setup(ctypes.byref(grid), W * n, self._ptr(s_dev), self._ptr(P.cell),
                                     self._ptr(P.lam), self.stream)
        _cabi.check(rc, "sdp_cell_setup")
        P.g = self.to_device(g_arr.reshape(-1)) if n else torch.zeros(1, dtype=torch.float64, device=self.device)
        P.p = self.to_device(w_proba)
        if world > 1:
            # every rank keeps the W table entries of relative DP's reference state (the
            # fused backup + shift kernel recomputes that state's value in every block)
            ref_flat = int(np.ravel_multi_index(solver._state_ref_ind, state_dims))
            rc_coords = np.stack([np.broadcast_to(self._as_full(c, full), full).reshape(n_grid, W)[ref_flat]
                                  for c in x_next])                       # [d][W]
            s_ref = self.to_device(np.ascontiguousarray(rc_coords))
            P.ref_cell = torch.empty(W, dtype=torch.int32, device=self.device)
            P.ref_lam = torch.empty(W * nb_state, dtype=torch.float64, device=self.device)
            rc = self.lib.sdp_cell_setup(ctypes.byref(grid), W, self._ptr(s_ref), self._ptr(P.ref_cell),
                                         self._ptr(P.ref_lam), self.stream)
            _cabi.check(rc, "sdp_cell_setup")
            g_full = self._as_full(g_k, full)
            if g_per_w:
                P.ref_g = self.to_device(np.ascontiguousarray(
                    np.broadcast_to(g_full, full).reshape(n_grid, W)[ref_flat]))
            else:
                P.ref_g = self.to_device(np.ascontiguousarray(
                    np.broadcast_to(g_full, state_dims + (1,)).reshape(n_grid)[ref_flat:ref_flat + 1]))
        return P

    @staticmethod
    def _as_full(a, full):
        """dyn/cost output as an fp64 array of the rank of `full` (leading axes of size 1 added)"""
        a = np.asarray(a)
        if a.dtype != np.float64:
            a = a.astype(float)
        return a.reshape((1,) * (len(full) - a.ndim) + a.shape)

    def policy_eval(self, P, J_a, J_b, n_iter, rel_dp, ref_index, J_ref_hist):
        """n_iter fixed-policy backups, ping-pong between J_a and J_b (device fp64
        [n_grid]).  Returns the tensor holding the final value function."""
        n_grid = J_a.numel()
        self.flush_exchange()
        if self.coll.world == 1:
            rc = self.lib.sdp_policy_eval(ctypes.byref(P.grid), P.W, P.g_per_w, self._ptr(P.p),
                                          self._ptr(P.cell), self._ptr(P.lam), P.lam_plane,
                                          self._ptr(P.g), P.n_states, 0, n_grid,
                                          self._ptr(J_a), self._ptr(J_b), int(n_iter),
                                          1 if rel_dp else 0, int(ref_index),
                                          self._ptr(J_ref_hist) if rel_dp else ctypes.c_void_p(0),
                                          self.stream)
            _cabi.check(rc, "sdp_policy_eval")
            return J_a if n_iter % 2 == 0 else J_b
        cur, nxt = J_a, J_b
        sb, n = P.state_begin, P.n_states
        px = self._peer.get(n_grid)
        if px is not None and px.index_of(J_a) is not None and px.index_of(J_b) is not None:
            # fused backup + all-gather over peer memory: the kernel stores the slab's new
            # values into every rank's buffer and publishes an epoch (no NCCL call)
            for k in range(n_iter):
                k_new = px.index_of(nxt)
                null = ctypes.c_void_p(0)
                rc = self.lib.sdp_policy_eval_p2p(
                    ctypes.byref(P.grid), P.W, P.g_per_w, self._ptr(P.p), self._ptr(P.cell),
                    self._ptr(P.lam), P.lam_plane, self._ptr(P.g), n, sb, n_grid, self._ptr(cur),
                    ctypes.byref(px.peers[k_new]),
                    self._ptr(P.ref_cell) if rel_dp else null, self._ptr(P.ref_lam) if rel_dp else null,
                    self._ptr(P.ref_g) if rel_dp else null,
                    ctypes.c_void_p(J_ref_hist.data_ptr() + 8 * k) if rel_dp else null, self.stream)
                _cabi.check(rc, "sdp_policy_eval_p2p")
                rc = self.lib.sdp_p2p_wait(ctypes.byref(px.peers[k_new]), self.stream)
                _cabi.check(rc, "sdp_p2p_wait")
                cur, nxt = nxt, cur
            return cur
        for k in range(n_iter):
            rc = self.lib.sdp_policy_eval(ctypes.byref(P.grid), P.W, P.g_per_w, self._ptr(P.p),
                                          self._ptr(P.cell), self._ptr(P.lam), P.lam_plane,
                                          self._ptr(P.g), n, sb, n_grid,
                                          self._ptr(cur), self._ptr(nxt), 1, 0, 0,
                                          ctypes.c_void_p(0), self.stream)
            _cabi.check(rc, "sdp_policy_eval")
            self.coll.all_gather_slabs(nxt[sb:sb + n].clone(), P.bounds, out=nxt)
            if rel_dp:
                ref_ptr = ctypes.c_void_p(J_ref_hist.data_ptr() + 8 * k)
                rc = self.lib.sdp_rel_shift(self._ptr(nxt), n_grid, int(ref_index), ref_ptr, self.stream)
                _cabi.check(rc, "sdp_rel_shift")
            cur, nxt = nxt, cur
        return cur

    # -- forward operator (distribution propagation) ----------------------
    def build_forward(self, P):
        """The transposed operator mu <- P^T mu of the policy tables `P` (sdp_forward_build):
        CSR by destination, g_bar, piece index of the long rows.  One rank only."""
        torch = _torch()
        if self.coll.world > 1 or P.n_states != int(np.prod(P.grid.order[:P.grid.d])):
            raise NotImplementedError(
                "distribution propagation runs on one rank: the transposed operator of a slab needs "
                "the sources of the other slabs (not implemented)")
        n = P.n_states
        nnz, max_pieces, build_b, step_d = (ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int64(),
                                            ctypes.c_int64())
        rc = self.lib.sdp_forward_sizes(P.grid.d, P.W, n, ctypes.byref(nnz), ctypes.byref(max_pieces),
                                        ctypes.byref(build_b), ctypes.byref(step_d))
        _cabi.check(rc, "sdp_forward_sizes")
        F = _cabi.SdpForwardOp()
        F.n, F.nnz, F.max_pieces = n, nnz.value, max_pieces.value
        dev = self.device
        bufs = {"row_ptr": torch.empty(n + 1, dtype=torch.int64, device=dev),
                "src": torch.empty(nnz.value, dtype=torch.int32, device=dev),
                "coef": torch.empty(nnz.value, dtype=torch.float64, device=dev),
                "gbar": torch.empty(n, dtype=torch.float64, device=dev),
                "piece_first": torch.empty(n + 1, dtype=torch.int64, device=dev),
                "piece_row": torch.empty(max_pieces.value, dtype=torch.int32, device=dev)}
        for name, t in bufs.items():
            setattr(F, name, t.data_ptr())
        # torch's caching allocator hands out 512-byte aligned blocks
        scratch = torch.empty(build_b.value, dtype=torch.uint8, device=dev)
        rc = self.lib.sdp_forward_build(ctypes.byref(P.grid), P.W, P.g_per_w, self._ptr(P.p), self._ptr(P.cell),
                                        self._ptr(P.lam), P.lam_plane, self._ptr(P.g), ctypes.byref(F),
                                        self._ptr(scratch), build_b.value, self.stream)
        _cabi.check(rc, "sdp_forward_build")
        F.n_pieces = int(bufs["piece_first"][n].item())      # sizes the piece pass of every step
        del scratch
        F.bufs = bufs
        F.step_scratch = torch.empty(step_d.value, dtype=torch.float64, device=dev)
        return F

    def forward_steps(self, F, mu_a, mu_b, n_steps, cost_out, resid_out=None, hist=None):
        """n_steps applications of P^T, ping-pong between mu_a (mu_0) and mu_b (device fp64 [n]);
        cost_out[k] = <mu_k, g_bar>, resid_out[0] = sum |mu_n - mu_{n-1}|, hist[k] = mu_k
        (device [(n_steps+1)*n]) when given.  Returns the tensor holding mu_n."""
        rc = self.lib.sdp_forward_steps(ctypes.byref(F), self._ptr(mu_a), self._ptr(mu_b), int(n_steps),
                                        self._ptr(cost_out), self._ptr(resid_out), self._ptr(hist),
                                        self._ptr(F.step_scratch), self.stream)
        _cabi.check(rc, "sdp_forward_steps")
        return mu_a if n_steps % 2 == 0 else mu_b

    def stationary(self, F, mu0, tol, max_iter, check_every):
        """Power iteration mu <- P^T mu from the host array mu0: launches of `check_every` steps
        (fewer for the last), one residual read back after each.  Returns (pi device tensor,
        steps done, residuals, converged)."""
        torch = _torch()
        mu_a = self.to_device(np.ascontiguousarray(mu0, dtype=np.float64).reshape(-1))
        mu_b = torch.empty_like(mu_a)
        cost = torch.empty(max(check_every, 1), dtype=torch.float64, device=self.device)
        resid = torch.zeros(1, dtype=torch.float64, device=self.device)
        residuals, done, converged = [], 0, False
        while done < max_iter:
            k = min(check_every, max_iter - done)
            mu_n = self.forward_steps(F, mu_a, mu_b, k, cost, resid)
            if mu_n is mu_b:
                mu_a, mu_b = mu_b, mu_a
            done += k
            r = float(resid.cpu().numpy()[0])
            residuals.append(r)
            if r <= tol:
                converged = True
                break
        return mu_a, done, residuals, converged

    # -- sample paths (Monte-Carlo trajectories) -------------------------
    def chain_tables(self, P):
        """The sampler's view of the policy tables `P` (sdp_chain_pack): one packed record per
        (x, w) and the cumulative node probabilities.  One rank only."""
        torch = _torch()
        if self.coll.world > 1 or P.n_states != int(np.prod(P.grid.order[:P.grid.d])):
            raise NotImplementedError(
                "path sampling runs on one rank: a path leaves the slab of its rank (not implemented)")
        n, d = P.n_states, P.grid.d
        C = ChainTables()
        C.grid, C.W, C.n = P.grid, P.W, n
        C.rec = torch.empty(n * P.W * _cabi.chain_rec(d), dtype=torch.float64, device=self.device)
        rc = self.lib.sdp_chain_pack(ctypes.byref(P.grid), P.W, P.g_per_w, self._ptr(P.cell), self._ptr(P.lam),
                                     P.lam_plane, self._ptr(P.g), n, self._ptr(C.rec), self.stream)
        _cabi.check(rc, "sdp_chain_pack")
        C.cdf = self.to_device(np.cumsum(P.p.cpu().numpy()))
        return C

    def chain_sample(self, C, state, total, hit, n_steps, step0, seed, fresh, counters, start_cdf=None,
                     target=None, rec_steps=None, rec_out=None):
        """Advance the paths (device state int32 / total fp64 / hit int32 [M]) by n_steps steps from
        global step step0 (sdp_chain_sample).  fresh: start at step0 from `state`, or from a state
        drawn with `start_cdf`; otherwise resume.  target: device uint32 bit mask; rec_steps: device
        int32 (increasing), rec_out [len(rec_steps) * M]; counters: device uint64 [2] (clamped, NaN
        transitions), accumulated."""
        n_rec = 0 if rec_steps is None else int(rec_steps.numel())
        rc = self.lib.sdp_chain_sample(ctypes.byref(C.grid), C.W, self._ptr(C.cdf), self._ptr(C.rec),
                                       int(state.numel()), int(n_steps), int(step0), int(seed), 1 if fresh else 0,
                                       self._ptr(start_cdf), self._ptr(target), self._ptr(rec_steps), n_rec,
                                       self._ptr(state), self._ptr(total), self._ptr(hit), self._ptr(rec_out),
                                       self._ptr(counters), self.stream)
        _cabi.check(rc, "sdp_chain_sample")

    # -- interpolation ----------------------------------------------------
    def interp(self, grid, values, s):
        """values: host (n_v, n_grid); s: host (d, n_s) -> host (n_v, n_s).
        fp64 or fp32 according to values.dtype."""
        torch = _torch()
        f32 = values.dtype == np.float32
        n_v, n_s = values.shape[0], s.shape[1]
        v_dev = self.to_device(values)
        s_dev = self.to_device(s)
        out = torch.empty((n_v, n_s), dtype=torch.float32 if f32 else torch.float64, device=self.device)
        fn = self.lib.sdp_interp_f32 if f32 else self.lib.sdp_interp
        rc = fn(ctypes.byref(grid), n_v, self._ptr(v_dev), n_s, self._ptr(s_dev), self._ptr(out), self.stream)
        _cabi.check(rc, "sdp_interp")
        return out.cpu().numpy()
