"""ctypes binding of libsdp_b200.so (C ABI declared in include/sdp_b200.h).

The library is the product's only compute path.  There is NO fallback: if the
shared object cannot be loaded, or an entry point returns an error, a
`SdpLibraryError` is raised.  torch is used by the callers only to own device
buffers; this module passes raw device pointers and the raw stream handle.
"""
import ctypes
import os

import numpy as np

SDP_MAX_D = 4
SDP_MAX_C = 4
SDP_ABI_VERSION = 10
LAYOUT_CONTROL_MINOR = 0   # "A": [state][w][u]
LAYOUT_STATE_MINOR = 1     # "B": [tile of 32 states][u][w][lane]
LAYOUT_CONTROL_MINOR_FACTORED = 2   # "AF": (x,u) part [state][Upad] + (x,w) part [state][W]
LAYOUT_STATE_MINOR_FACTORED = 3     # "BF": (x,u) part [tile][u][lane] + (x,w) part [tile][w][lane]
LAYOUT_COLUMN_FACTORED = 4          # "CF": BF tables over column-major tiles, inner interpolation shared per column
COLUMN_MAX_SMEM_BYTES = 200 * 1024  # CF: 8 * column_pitch(order[0], W) bytes of shared memory per CTA


def column_pitch(rows, W, pairs=False):
    """SDP_COLUMN_PITCH / SDP_COLUMN_PITCH2: doubles per column table of layout CF"""
    if pairs:
        return (rows * (W | 1) + (rows >> 1) + 10 + 1) & ~1
    return (rows * (W | 1) + 9 + 1) & ~1


FACTORED_MAX_W_REG = 9     # BF keeps a lane's w-part in registers
FACTORED_MAX_W_SMEM = 128  # AF keeps a state's w-part in shared memory

_HERE = os.path.dirname(os.path.abspath(__file__))
# SDP_B200_LIB: developer override (kernel variants built side by side for tuning runs)
LIB_PATH = os.environ.get("SDP_B200_LIB") or os.path.join(_HERE, "_lib", "libsdp_b200.so")


class SdpLibraryError(RuntimeError):
    """The CUDA extension is missing, stale, or one of its entry points failed."""


class SdpGrid(ctypes.Structure):
    _fields_ = [("d", ctypes.c_int32),
                ("order", ctypes.c_int32 * SDP_MAX_D),
                ("smin", ctypes.c_double * SDP_MAX_D),
                ("smax", ctypes.c_double * SDP_MAX_D)]


class SdpTables(ctypes.Structure):
    _fields_ = [("cell", ctypes.c_void_p),
                ("lam", ctypes.c_void_p),
                ("lam_plane", ctypes.c_int64),
                ("g", ctypes.c_void_p),
                ("g_per_w", ctypes.c_int32),
                ("W", ctypes.c_int32),
                ("expect", ctypes.c_int32),
                ("layout", ctypes.c_int32),
                ("p", ctypes.c_void_p),
                ("items", ctypes.c_void_p),
                ("n_items", ctypes.c_int64),
                ("item_begin", ctypes.c_void_p),
                ("n_states", ctypes.c_int64),
                ("U", ctypes.c_void_p),
                ("u_mask", ctypes.c_int32),
                ("col_pairs", ctypes.c_int32),
                ("cell_w", ctypes.c_void_p),
                ("lam_w", ctypes.c_void_p),
                ("lam_w_plane", ctypes.c_int64),
                ("p_host", ctypes.c_void_p),
                ("n_cols", ctypes.c_int32),
                ("tiles_per_col", ctypes.c_int32),
                ("seg_begin", ctypes.c_void_p),
                ("n_segs", ctypes.c_int64),
                ("col_table", ctypes.c_void_p),
                ("run_end", ctypes.c_void_p),
                ("col_table_ready", ctypes.c_int32),
                ("col_launch_hint", ctypes.c_int32),
                ("item_order", ctypes.c_void_p),
                ("pos_row", ctypes.c_void_p),
                ("col_bound", ctypes.c_void_p)]


SDP_MAX_PEERS = 8


class SdpPeers(ctypes.Structure):
    _fields_ = [("world", ctypes.c_int32),
                ("rank", ctypes.c_int32),
                ("J", ctypes.c_void_p * SDP_MAX_PEERS),
                ("flags", ctypes.c_void_p * SDP_MAX_PEERS),
                ("epoch", ctypes.c_void_p),
                ("done", ctypes.c_void_p),
                ("A", ctypes.c_void_p * SDP_MAX_PEERS)]


class SdpForwardOp(ctypes.Structure):
    """forward (adjoint) operator of a fixed policy: CSR by destination (sdp_forward_*)"""
    _fields_ = [("n", ctypes.c_int64),
                ("nnz", ctypes.c_int64),
                ("row_ptr", ctypes.c_void_p),
                ("src", ctypes.c_void_p),
                ("coef", ctypes.c_void_p),
                ("gbar", ctypes.c_void_p),
                ("piece_first", ctypes.c_void_p),
                ("piece_row", ctypes.c_void_p),
                ("max_pieces", ctypes.c_int64),
                ("n_pieces", ctypes.c_int64)]


FWD_PIECE = 1024   # SDP_FWD_PIECE: entries per piece of a long row of the forward operator
CHAIN_INIT_STEP = 0xFFFFFFFF   # SDP_CHAIN_INIT_STEP: Philox step word of the initial-state draws


def chain_rec(d):
    """SDP_CHAIN_REC: doubles per packed (x, w) record of sdp_chain_sample"""
    return 2 * ((d + 3) // 2)


# numpy mirrors of the per-state descriptor and the work item (host-built arrays
# uploaded verbatim; layouts must match the C structs, checked by the tests)
STATE_DESC_DTYPE = np.dtype([("entry_off", np.int64),
                             ("g_off", np.int64),
                             ("src", np.int64, (SDP_MAX_D + 1,)),
                             ("cs", np.int32, (SDP_MAX_D + 1, SDP_MAX_C)),
                             ("ws", np.int32, (SDP_MAX_D + 1,)),
                             ("npts", np.int32, (SDP_MAX_C,)),
                             ("U", np.int32),
                             ("Upad", np.int32)], align=True)
ITEM_DTYPE = np.dtype([("entry_base", np.int64),
                       ("g_base", np.int64),
                       ("Upad", np.int32),
                       ("u_begin", np.int32),
                       ("u_count", np.int32),
                       ("state", np.int32)], align=True)
assert STATE_DESC_DTYPE.itemsize == 184, STATE_DESC_DTYPE.itemsize
assert ITEM_DTYPE.itemsize == 32, ITEM_DTYPE.itemsize

_vp = ctypes.c_void_p
_i32 = ctypes.c_int32
_i64 = ctypes.c_int64
_gp = ctypes.POINTER(SdpGrid)

# name -> (restype, argtypes); every symbol include/sdp_b200.h declares
SIGNATURES = {
    "sdp_version": (ctypes.c_int, []),
    "sdp_last_error": (ctypes.c_char_p, []),
    "sdp_launch_count": (_i64, []),
    "sdp_last_kernel": (ctypes.c_char_p, []),
    "sdp_set_option": (ctypes.c_int, [ctypes.c_char_p, ctypes.c_int]),
    "sdp_col_prune_counts": (ctypes.c_int, [ctypes.POINTER(_i64), ctypes.POINTER(_i64)]),
    "sdp_cell_setup": (ctypes.c_int, [_gp, _i64, _vp, _vp, _vp, _vp]),
    "sdp_build_tables": (ctypes.c_int, [_gp, _i32, _i32, _i64, _vp, _vp, _vp, _vp, _i64, _vp,
                                        _i32, _vp]),
    "sdp_build_tables_tiled": (ctypes.c_int, [_gp, _i32, _i32, _i64, _vp, _vp, _i64, _vp, _vp, _vp,
                                              _i32, _vp, _vp, _i64, _vp, _vp]),
    "sdp_build_tables_factored": (ctypes.c_int, [_gp, _i32, _i32, _i64, _vp, _vp, _vp, _vp, _i64, _vp,
                                                 _i32, _vp, _vp, _i64, _vp]),
    "sdp_build_tables_factored_tiled": (ctypes.c_int, [_gp, _i32, _i32, _i64, _vp, _vp, _i64, _vp, _vp,
                                                       _i32, _vp, _vp, _i64, _vp, _vp, _vp, _i64, _vp]),
    "sdp_sweep": (ctypes.c_int, [_gp, ctypes.POINTER(SdpTables), _vp, _vp, _vp, _vp, _vp, _vp]),
    "sdp_column_table": (ctypes.c_int, [_gp, ctypes.POINTER(SdpTables), _vp, _vp]),
    "sdp_sweep_partials": (ctypes.c_int, [_gp, ctypes.POINTER(SdpTables), _vp, _vp, _vp, _vp]),
    "sdp_sweep_finalize": (ctypes.c_int, [ctypes.POINTER(SdpTables), _vp, _vp, _vp, _vp, _vp]),
    "sdp_sweep_finalize_p2p": (ctypes.c_int, [ctypes.POINTER(SdpTables), _vp, _vp, _vp,
                                              ctypes.POINTER(SdpPeers), _i64, _vp]),
    "sdp_sweep_finalize_p2p_cols": (ctypes.c_int, [ctypes.POINTER(SdpTables), _vp, _vp, _vp,
                                                   ctypes.POINTER(SdpPeers), _i64, _i64, _vp]),
    "sdp_p2p_wait": (ctypes.c_int, [ctypes.POINTER(SdpPeers), _vp]),
    "sdp_sweep_partials_after": (ctypes.c_int, [_gp, ctypes.POINTER(SdpTables), _vp, _vp, _vp,
                                                ctypes.POINTER(SdpPeers), _vp]),
    "sdp_p2p_barrier": (ctypes.c_int, [ctypes.POINTER(SdpPeers), _vp]),
    "sdp_p2p_broadcast": (ctypes.c_int, [_vp, _i64, _i64, ctypes.POINTER(SdpPeers), _vp]),
    "sdp_policy_eval": (ctypes.c_int, [_gp, _i32, _i32, _vp, _vp, _vp, _i64, _vp, _i64, _i64, _i64,
                                       _vp, _vp, _i32, _i32, _i64, _vp, _vp]),
    "sdp_policy_eval_p2p": (ctypes.c_int, [_gp, _i32, _i32, _vp, _vp, _vp, _i64, _vp, _i64, _i64, _i64,
                                           _vp, ctypes.POINTER(SdpPeers), _vp, _vp, _vp, _vp, _vp]),
    "sdp_forward_sizes": (ctypes.c_int, [_i32, _i32, _i64, _vp, _vp, _vp, _vp]),
    "sdp_forward_build": (ctypes.c_int, [_gp, _i32, _i32, _vp, _vp, _vp, _i64, _vp,
                                         ctypes.POINTER(SdpForwardOp), _vp, _i64, _vp]),
    "sdp_forward_steps": (ctypes.c_int, [ctypes.POINTER(SdpForwardOp), _vp, _vp, _i32, _vp, _vp, _vp, _vp,
                                         _vp]),
    "sdp_chain_pack": (ctypes.c_int, [_gp, _i32, _i32, _vp, _vp, _i64, _vp, _i64, _vp, _vp]),
    "sdp_chain_sample": (ctypes.c_int, [_gp, _i32, _vp, _vp, _i64, _i32, _i64, ctypes.c_uint64, _i32, _vp, _vp,
                                        _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sdp_first_passage": (ctypes.c_int, [_gp, _i32, _i32, _vp, _vp, _vp, _i64, _vp, _i64, _vp, _i32, _vp, _vp, _i32,
                                         _vp, _vp, _vp, _vp]),
    "sdp_cost_moments": (ctypes.c_int, [_gp, _i32, _i32, _vp, _vp, _vp, _i64, _vp, _i64, _vp, _i32, _vp, _vp, _i32,
                                        _vp, _vp, _vp, _vp]),
    "sdp_policy_values": (ctypes.c_int, [_i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "sdp_sweep_finalize_cols": (ctypes.c_int, [ctypes.POINTER(SdpTables), _vp, _vp, _vp, _vp, _i64, _i64,
                                               _i32, _vp, _vp, _vp, _vp, _i32, _vp]),
    "sdp_memcpy_2d": (ctypes.c_int, [_vp, _i64, _vp, _i64, _i64, _i64, _vp]),
    "sdp_rel_shift": (ctypes.c_int, [_vp, _i64, _i64, _vp, _vp]),
    "sdp_supnorm_diff": (ctypes.c_int, [_vp, _vp, _i64, _vp, _vp]),
    "sdp_interp": (ctypes.c_int, [_gp, _i64, _vp, _i64, _vp, _vp, _vp]),
    "sdp_interp_f32": (ctypes.c_int, [_gp, _i64, _vp, _i64, _vp, _vp, _vp]),
    "sdp_interp_host": (ctypes.c_int, [_gp, _i64, _vp, _i64, _vp, _vp]),
    "sdp_interp_host_f32": (ctypes.c_int, [_gp, _i64, _vp, _i64, _vp, _vp]),
}

_lib = None


def load_library(path=None):
    """Load (once) and type the shared library.  Raises SdpLibraryError."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise SdpLibraryError(
            "CUDA extension not built: %s is missing. Run `python -m stodynprog_b200.build` "
            "(or __graft_entry__.build()); there is no CPU fallback." % p)
    try:
        lib = ctypes.CDLL(p)
    except OSError as e:
        raise SdpLibraryError("cannot load %s: %s" % (p, e))
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:
            raise SdpLibraryError("%s does not export %s (stale build?)" % (p, name))
        fn.restype = res
        fn.argtypes = args
    if lib.sdp_version() != SDP_ABI_VERSION:
        raise SdpLibraryError("ABI version mismatch: library %d, binding %d"
                              % (lib.sdp_version(), SDP_ABI_VERSION))
    if path is None:
        _lib = lib
    return lib


def check(rc, what):
    """Raise on a negative return code of an entry point."""
    if rc != 0:
        msg = load_library().sdp_last_error()
        raise SdpLibraryError("%s failed (code %d): %s"
                              % (what, rc, msg.decode("utf-8", "replace") if msg else ""))


def make_grid(state_grid):
    """SdpGrid from a list of 1-D grids: smin = g[0], smax = g[-1], order = len(g)
    (what MlinInterpolator.__init__ keeps, reference stodynprog.py:261-265)."""
    d = len(state_grid)
    if not 1 <= d <= SDP_MAX_D:
        raise ValueError("state dimension %d not supported by the CUDA kernels (1..%d)"
                         % (d, SDP_MAX_D))
    g = SdpGrid()
    g.d = d
    for k, ax in enumerate(state_grid):
        g.order[k] = len(ax)
        g.smin[k] = float(ax[0])
        g.smax[k] = float(ax[-1])
    return g


def launch_count():
    return int(load_library().sdp_launch_count())


def last_kernel():
    """the streaming kernel this thread's last sweep launched, as the library names it"""
    name = load_library().sdp_last_kernel()
    return name.decode("utf-8", "replace") if name else ""
