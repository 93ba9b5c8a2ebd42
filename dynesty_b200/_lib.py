"""ctypes binding of libb200nest.so (C ABI: include/b200nest.h).

There is NO CPU fallback: if the library is missing or no CUDA device is
available every entry point raises ``B200Unavailable``.
"""
import ctypes as C
import itertools
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIBPATH = os.path.join(HERE, 'libb200nest.so')

PTR_HOST, PTR_DEVICE = 0, 1
DIM_PERIODIC, DIM_REFLECTIVE = 1, 2
PRIOR_IDENTITY, PRIOR_UNIFORM, PRIOR_NORMAL_PPF = 0, 1, 2
LIKE_GAUSS_PREC, LIKE_GAUSS_DIAG, LIKE_EGGBOX, LIKE_SHELLS, LIKE_REGION2D = 0, 1, 2, 3, 4
WARN_IDENTITY_FALLBACK, WARN_DOUBLING, WARN_Q0_SLACK, WARN_UNIF_INEFFICIENT = 1, 2, 4, 8

(OK, ERR_CUDA, ERR_ARG, ERR_SINGLE_POINT, ERR_SINGULAR, ERR_ELL_INIT, ERR_INVALID_REGION,
 ERR_Q0, ERR_SLICE_FAIL, ERR_NOMEM, ERR_UNSUPPORTED, ERR_TOO_MANY_ELLS, ERR_PEER, ERR_PLATEAU) = range(14)
PEER_HANDLE_BYTES, MAX_PEERS = 64, 8


class B200Unavailable(RuntimeError):
    """libb200nest.so / a CUDA device is missing.  The B200 path has no CPU fallback."""


class ModelDesc(C.Structure):
    _fields_ = [('ndim', C.c_int32), ('prior_kind', C.c_int32), ('like_kind', C.c_int32),
                ('reserved', C.c_int32), ('prior_p0', C.c_void_p), ('prior_p1', C.c_void_p),
                ('like_vec0', C.c_void_p), ('like_vec1', C.c_void_p), ('like_mat', C.c_void_p),
                ('like_s0', C.c_double), ('like_s1', C.c_double), ('like_s2', C.c_double)]


class ChainArgs(C.Structure):
    _fields_ = [('nchain', C.c_int64), ('ndim', C.c_int32), ('ncdim', C.c_int32),
                ('model_id', C.c_int32), ('reserved', C.c_int32), ('u0', C.c_void_p),
                ('ell', C.c_void_p), ('dimflags', C.c_void_p), ('loglstar', C.c_double),
                ('scale', C.c_double), ('seed', C.c_uint64), ('chain0', C.c_uint64)]


class NsConfig(C.Structure):
    _fields_ = [('nlive', C.c_int32), ('ndim', C.c_int32), ('ncdim', C.c_int32), ('batch', C.c_int32),
                ('sampler', C.c_int32), ('steps', C.c_int32), ('model_id', C.c_int32),
                ('strict_contains', C.c_int32), ('facc', C.c_double), ('dlogz', C.c_double),
                ('maxiter', C.c_int64), ('maxcall', C.c_int64), ('update_interval', C.c_int64),
                ('seed', C.c_uint64), ('chain0', C.c_uint64), ('dimflags', C.c_void_p),
                ('unit_cube_phase', C.c_int32), ('use_logl_max', C.c_int32), ('first_min_ncall', C.c_int64),
                ('first_min_eff', C.c_double), ('logl_max', C.c_double), ('it0', C.c_int64)]


class NsStatus(C.Structure):
    _fields_ = [('it', C.c_int64), ('ncall', C.c_int64), ('rounds', C.c_int64), ('logz', C.c_double),
                ('logvol', C.c_double), ('loglstar', C.c_double), ('lmax', C.c_double),
                ('delta_logz', C.c_double), ('scale', C.c_double), ('done', C.c_int32),
                ('need_bound', C.c_int32), ('doubling', C.c_int32), ('error', C.c_int32),
                ('ncall_last_update', C.c_int64)]


# every symbol include/b200nest.h declares: (restype, argtypes)
_P, _I, _L, _D, _U64 = C.c_void_p, C.c_int32, C.c_int64, C.c_double, C.c_uint64
SYMBOLS = {
    'b2n_init': (C.c_int, [C.c_int, C.POINTER(_P)]),
    'b2n_free': (None, [_P]),
    'b2n_set_stream': (C.c_int, [_P, _P]),
    'b2n_set_pointer_mode': (C.c_int, [_P, C.c_int]),
    'b2n_synchronize': (C.c_int, [_P]),
    'b2n_set_chain_pack': (C.c_int, [_P, _I]),
    'b2n_set_start_rows': (C.c_int, [_P, _P, C.c_int64]),
    'b2n_debug_launch_rate': (C.c_int, [_P, _I, C.POINTER(_D)]),
    'b2n_strerror': (C.c_char_p, [C.c_int]),
    'b2n_last_error': (C.c_char_p, [_P]),
    'b2n_version': (C.c_char_p, []),
    'b2n_launch_count': (C.c_int64, [_P]),
    'b2n_set_timing': (C.c_int, [_P, C.c_int]),
    'b2n_last_kernel_ms': (C.c_double, [_P]),
    'b2n_model_create': (C.c_int, [_P, C.POINTER(ModelDesc), C.POINTER(_I)]),
    'b2n_model_eval': (C.c_int, [_P, _I, _P, _L, _P, _P]),
    'b2n_membership': (C.c_int, [_P, _P, _L, _I, _P, _P, _I, _I, _P, _P, _P]),
    'b2n_bounding_ellipsoid': (C.c_int, [_P, _P, _L, _I, _P, _P, _P, _P, _P, _P, _P]),
    'b2n_multi_decompose': (C.c_int, [_P, _P, _L, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    'b2n_moments': (C.c_int, [_P, _P, _L, _I, _P, _P]),
    'b2n_improve_covar': (C.c_int, [_P, _P, _I, _P, _P, _P, _P, _P]),
    'b2n_fp64_peak': (C.c_int, [_P, _I, _I, C.POINTER(_D), C.POINTER(_D)]),
    'b2n_scale_to_logvol': (C.c_int, [_P, _I, _I, _P, _P, _P, _P, _P, _P]),
    'b2n_bootstrap_expand': (C.c_int, [_P, _P, _L, _I, _I, _I, _U64, _U64, _P]),
    'b2n_friends_update': (C.c_int, [_P, _P, _L, _I, _I, _I, _P, _I, _U64, _U64, _P, _P, _P, _P, _P, _P, _P]),
    'b2n_friends_set': (C.c_int, [_P, _I, _P, _L, _I, _P, _P]),
    'b2n_friends_overlap': (C.c_int, [_P, _P, _L, _I, _P]),
    'b2n_friends_unif_batch': (C.c_int, [_P, C.POINTER(ChainArgs), _P, _P, _P, _P, _P, _P]),
    'b2n_bound_set': (C.c_int, [_P, _I, _I, _P, _P, _P, _P]),
    'b2n_rwalk_batch': (C.c_int, [_P, C.POINTER(ChainArgs), _I, _P, _P, _P, _P, _P, _P]),
    'b2n_rslice_batch': (C.c_int, [_P, C.POINTER(ChainArgs), _I, _I, _P, _P, _P, _P, _P, _P, _P]),
    'b2n_slice_batch': (C.c_int, [_P, C.POINTER(ChainArgs), _I, _I, _P, _P, _P, _P, _P, _P, _P]),
    'b2n_unitcube_batch': (C.c_int, [_P, C.POINTER(ChainArgs), _P, _P, _P, _P, _P]),
    'b2n_unif_batch': (C.c_int, [_P, C.POINTER(ChainArgs), _P, _P, _P, _P, _P, _P]),
    'b2n_peer_export': (C.c_int, [_P, _U64, _P]),
    'b2n_peer_import': (C.c_int, [_P, _I, _I, _P]),
    'b2n_peer_import_raw': (C.c_int, [_P, _I, _I, C.POINTER(_P)]),
    'b2n_peer_rows': (C.c_int, [_P, _L, _L]),
    'b2n_peer_result': (C.c_int, [_P, C.POINTER(_P), C.POINTER(_U64)]),
    'b2n_peer_read': (C.c_int, [_P, _U64, _P, _U64]),
    'b2n_peer_check': (C.c_int, [_P]),
    'b2n_peer_window_bytes': (_U64, [_L, _I]),
    'b2n_ns_create': (C.c_int, [_P, C.POINTER(NsConfig), _L]),
    'b2n_ns_destroy': (C.c_int, [_P]),
    'b2n_ns_set_state': (C.c_int, [_P, _P, _P, _P, _D, _D, _D, _L, _L, _D]),
    'b2n_ns_run': (C.c_int, [_P, _I, _I, C.POINTER(NsStatus)]),
    'b2n_ns_status_get': (C.c_int, [_P, C.POINTER(NsStatus)]),
    'b2n_ns_set_counters': (C.c_int, [_P, _L, _L, _I]),
    'b2n_ns_bound_updated': (C.c_int, [_P]),
    'b2n_ns_update_bound': (C.c_int, [_P, _I, _D, _P, _P, _P]),
    'b2n_ns_get_bound': (C.c_int, [_P, _I, _P, _P, _P, _P, _P, _P]),
    'b2n_ns_update_friends': (C.c_int, [_P, _I, _D, _I, _I, _P, _P, _P]),
    'b2n_ns_set_friends': (C.c_int, [_P, _I, _P, _P, _P, _P, _D]),
    'b2n_ns_get_friends': (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P]),
    'b2n_ns_reserve_dead': (C.c_int, [_P, _L]),
    'b2n_ns_get_live': (C.c_int, [_P, _P, _P, _P]),
    'b2n_ns_get_dead': (C.c_int, [_P, _L, _L, _P, _P, _P, _P, _P]),
}

_lib = None


def load():
    """dlopen the library and bind every declared symbol (no CUDA calls)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIBPATH):
        raise B200Unavailable(
            "%s not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  There is no CPU fallback." % LIBPATH)
    lib = C.CDLL(LIBPATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


_EXC = {
    ERR_ARG: ValueError, ERR_SINGLE_POINT: ValueError, ERR_SINGULAR: ValueError,
    ERR_ELL_INIT: RuntimeError, ERR_INVALID_REGION: RuntimeError, ERR_Q0: RuntimeError,
    ERR_SLICE_FAIL: RuntimeError, ERR_NOMEM: MemoryError, ERR_UNSUPPORTED: NotImplementedError,
    ERR_TOO_MANY_ELLS: RuntimeError, ERR_PEER: RuntimeError, ERR_PLATEAU: RuntimeError,
}


def ptr(a):
    """Address of a numpy array / torch tensor / int / None."""
    if a is None:
        return None
    if isinstance(a, int):
        return a
    if isinstance(a, np.ndarray):
        assert a.flags['C_CONTIGUOUS'], "array must be C-contiguous"
        return a.ctypes.data
    return a.data_ptr()      # torch tensor


def f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


_ctx_serial = itertools.count(1)


class Context:
    """Owns one b2n_ctx.  One per process / GPU is the normal case; several contexts on one GPU
    (each with its own stream and scratch memory) run concurrently -- ``dynesty_b200.replicas``."""

    def __init__(self, device=0):
        self.lib = load()
        self.serial = next(_ctx_serial)      # never reused, unlike id(): the key of per-context caches
        self.resident_key = None             # version token of the bound whose ellipsoids are resident (ops.bound_set)
        self.friends_key = None              # same for the resident RadFriends / SupFriends bound (ops.friends_set)
        h = C.c_void_p()
        st = self.lib.b2n_init(int(device), C.byref(h))
        if st != OK:
            raise B200Unavailable(
                "b2n_init(device=%d) failed: %s -- the B200 path needs a CUDA device; "
                "there is no CPU fallback" % (device, self.lib.b2n_strerror(st).decode()))
        self.h = h
        self.device = device
        self.mode = PTR_HOST

    def close(self):
        if getattr(self, 'h', None):
            self.lib.b2n_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, st):
        if st == OK:
            return
        msg = self.lib.b2n_strerror(st).decode()
        detail = self.lib.b2n_last_error(self.h).decode()
        if st == ERR_CUDA or detail:
            msg = "%s (%s)" % (msg, detail)
        raise _EXC.get(st, RuntimeError)(msg)

    def set_stream(self, stream):
        self.check(self.lib.b2n_set_stream(self.h, stream))

    def set_pointer_mode(self, mode):
        self.check(self.lib.b2n_set_pointer_mode(self.h, mode))
        self.mode = mode

    def set_chain_pack(self, chains_per_cta):
        self.check(self.lib.b2n_set_chain_pack(self.h, int(chains_per_cta)))

    def set_start_rows(self, idx_ptr, nrows):
        """the next rwalk call takes its start points as rows idx[q] of its u0 (= the whole live set)"""
        self.check(self.lib.b2n_set_start_rows(self.h, idx_ptr, int(nrows)))

    def synchronize(self):
        self.check(self.lib.b2n_synchronize(self.h))

    def set_timing(self, enabled):
        self.check(self.lib.b2n_set_timing(self.h, int(bool(enabled))))

    def last_kernel_ms(self):
        return float(self.lib.b2n_last_kernel_ms(self.h))

    def launch_count(self):
        return int(self.lib.b2n_launch_count(self.h))

    # ---- multi-GPU exchange windows (include/b200nest.h, "peer" section) ------------------
    def peer_window_bytes(self, total_rows, ndim):
        return int(self.lib.b2n_peer_window_bytes(int(total_rows), int(ndim)))

    def peer_export(self, nbytes):
        """Allocate this rank's exchange window; returns its 64-byte CUDA IPC handle."""
        buf = (C.c_ubyte * PEER_HANDLE_BYTES)()
        self.check(self.lib.b2n_peer_export(self.h, int(nbytes), C.cast(buf, C.c_void_p)))
        return bytes(buf)

    def peer_import(self, rank, world, handles):
        """Map the windows of all ranks (handles: world x 64 bytes, rank order)."""
        blob = b''.join(handles) if not isinstance(handles, (bytes, bytearray)) else bytes(handles)
        assert len(blob) == world * PEER_HANDLE_BYTES
        buf = (C.c_ubyte * len(blob)).from_buffer_copy(blob)
        self.check(self.lib.b2n_peer_import(self.h, int(rank), int(world), C.cast(buf, C.c_void_p)))

    def peer_import_raw(self, rank, world, windows):
        """Same for ranks that live in this process: device addresses of their windows."""
        arr = (C.c_void_p * world)(*[C.c_void_p(int(w)) for w in windows])
        self.check(self.lib.b2n_peer_import_raw(self.h, int(rank), int(world), arr))

    def peer_rows(self, row0, total_rows):
        self.check(self.lib.b2n_peer_rows(self.h, int(row0), int(total_rows)))

    def peer_result(self):
        """(window device address, byte offsets of u, v, logl, int0..int3) of the last gather-mode call."""
        w = C.c_void_p()
        off = (C.c_uint64 * 7)()
        self.check(self.lib.b2n_peer_result(self.h, C.byref(w), off))
        return int(w.value), [int(x) for x in off]

    def peer_read(self, offset, shape, dtype):
        """Synchronise and fetch an array that starts at byte `offset` of the own window."""
        a = np.empty(shape, dtype=dtype)
        self.check(self.lib.b2n_peer_read(self.h, int(offset), a.ctypes.data, a.nbytes))
        return a

    def peer_gathered(self, total_rows, ndim, names):
        """The complete outputs of the last gather-mode call, read from the own window:
        u, v, logl and the call's int32 outputs under `names` (argument order, None = skip)."""
        _, off = self.peer_result()
        o = dict(u=self.peer_read(off[0], (total_rows, ndim), np.float64),
                 v=self.peer_read(off[1], (total_rows, ndim), np.float64),
                 logl=self.peer_read(off[2], (total_rows,), np.float64))
        for k, nm in enumerate(names):
            if nm is not None:
                o[nm] = self.peer_read(off[3 + k], (total_rows,), np.uint32 if nm == 'flags' else np.int32)
        return o

    def peer_check(self):
        self.check(self.lib.b2n_peer_check(self.h))


_default_ctx = {}


def default_context(device=None):
    if device is None:
        device = int(os.environ.get('LOCAL_RANK', '0'))
    if device not in _default_ctx:
        _default_ctx[device] = Context(device)
    return _default_ctx[device]
