"""numpy-level wrappers of the C ABI (host-pointer mode).  Every function here is a
single C call; array-in/array-out, the reference's exceptions on failure."""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import ChainArgs, ptr, f64


def _ctx(ctx):
    return ctx if ctx is not None else _lib.default_context()


def model_eval(model, u, want_v=True, ctx=None):
    """(v, logl) for the rows of u (M, ndim)."""
    ctx = _ctx(ctx)
    u = f64(np.atleast_2d(u))
    M, n = u.shape
    v = np.empty((M, n)) if want_v else None
    logl = np.empty(M)
    ctx.check(ctx.lib.b2n_model_eval(ctx.h, model, ptr(u), M, ptr(v), ptr(logl)))
    return v, logl


def membership(x, ctrs, ams, strict=True, want_d2=False, ctx=None):
    """mask (M, K) bool, q (M,) int32 [, d2 (M, K)]  (bounding.py:502-523)."""
    ctx = _ctx(ctx)
    x = f64(np.atleast_2d(x))
    ctrs = f64(np.atleast_2d(ctrs))
    ams = f64(ams).reshape(ctrs.shape[0], ctrs.shape[1], ctrs.shape[1])
    M, n = x.shape
    K = ctrs.shape[0]
    mask = np.empty((M, K), dtype=np.uint8)
    q = np.empty(M, dtype=np.int32)
    d2 = np.empty((M, K)) if want_d2 else None
    ctx.check(ctx.lib.b2n_membership(ctx.h, ptr(x), M, n, ptr(ctrs), ptr(ams), K, int(bool(strict)),
                                     ptr(mask), ptr(q), ptr(d2)))
    out = (mask.astype(bool), q)
    return out + (d2,) if want_d2 else out


def bounding_ellipsoid(points, ctx=None):
    """dict(ctr, cov, am, axes, axlens, logvol, warn)  (bounding.py:1387-1461)."""
    ctx = _ctx(ctx)
    points = f64(points)
    N, n = points.shape
    o = dict(ctr=np.empty(n), cov=np.empty((n, n)), am=np.empty((n, n)), axes=np.empty((n, n)),
             axlens=np.empty(n))
    lv = np.empty(1)
    warn = C.c_uint32(0)
    ctx.check(ctx.lib.b2n_bounding_ellipsoid(ctx.h, ptr(points), N, n, ptr(o['ctr']), ptr(o['cov']),
                                             ptr(o['am']), ptr(o['axes']), ptr(o['axlens']), ptr(lv),
                                             C.addressof(warn)))
    o['logvol'] = float(lv[0])
    o['warn'] = warn.value
    return o


def multi_decompose(points, max_ells=None, ctx=None):
    """dict(nells, labels, ctrs, covs, ams, axes, axlens, logvols, warn)  (bounding.py:665-686)."""
    ctx = _ctx(ctx)
    points = f64(points)
    N, n = points.shape
    if max_ells is None:
        max_ells = max(1, N // max(2 * n, 1))
    K = int(max_ells)
    o = dict(labels=np.empty(N, dtype=np.int32), ctrs=np.empty((K, n)), covs=np.empty((K, n, n)),
             ams=np.empty((K, n, n)), axes=np.empty((K, n, n)), axlens=np.empty((K, n)),
             logvols=np.empty(K))
    nells = C.c_int32(0)
    warn = C.c_uint32(0)
    ctx.check(ctx.lib.b2n_multi_decompose(ctx.h, ptr(points), N, n, K, C.addressof(nells),
                                          ptr(o['labels']), ptr(o['ctrs']), ptr(o['covs']), ptr(o['ams']),
                                          ptr(o['axes']), ptr(o['axlens']), ptr(o['logvols']),
                                          C.addressof(warn)))
    k = nells.value
    for key in ('ctrs', 'covs', 'ams', 'axes', 'axlens', 'logvols'):
        o[key] = o[key][:k].copy()
    o['nells'] = k
    o['warn'] = warn.value
    return o


def moments(points, ctx=None):
    """(mean, cov) = (np.mean(points, 0), np.cov(points, rowvar=False)) of one shard of the live set."""
    ctx = _ctx(ctx)
    points = f64(points)
    N, n = points.shape
    mean, cov = np.empty(n), np.empty((n, n))
    ctx.check(ctx.lib.b2n_moments(ctx.h, ptr(points), N, n, ptr(mean), ptr(cov)))
    return mean, cov


def improve_covar(covar, ctx=None):
    """(good, cov, am, axes, warn) = improve_covar_mat(covar)  (bounding.py:1311-1384)."""
    ctx = _ctx(ctx)
    covar = f64(covar)
    n = covar.shape[0]
    cov, am, axes = np.empty((n, n)), np.empty((n, n)), np.empty((n, n))
    good, warn = C.c_int32(0), C.c_uint32(0)
    ctx.check(ctx.lib.b2n_improve_covar(ctx.h, ptr(covar), n, ptr(cov), ptr(am), ptr(axes), C.addressof(good),
                                        C.addressof(warn)))
    return bool(good.value), cov, am, axes, warn.value


def fp64_peak(kind, iters=20000, ctx=None):
    """Measured FP64 ceiling in TFLOP/s: kind 'fma' (vector pipe) or 'mma' (m8n8k4 tensor pipe)."""
    ctx = _ctx(ctx)
    t, ms = C.c_double(0.0), C.c_double(0.0)
    ctx.check(ctx.lib.b2n_fp64_peak(ctx.h, {'fma': 0, 'mma': 1}[kind], int(iters), C.byref(t), C.byref(ms)))
    return t.value, ms.value


def scale_to_logvol(covs, ams, axes, axlens, logvols, targets, ctx=None):
    """In-place Ellipsoid.scale_to_logvol on K stacked ellipsoids (bounding.py:242-276)."""
    ctx = _ctx(ctx)
    K, n = axlens.shape
    targets = f64(targets)
    for a in (covs, ams, axes, axlens, logvols):
        assert a.dtype == np.float64 and a.flags['C_CONTIGUOUS']
    ctx.check(ctx.lib.b2n_scale_to_logvol(ctx.h, K, n, ptr(covs), ptr(ams), ptr(axes), ptr(axlens),
                                          ptr(logvols), ptr(targets)))


def bootstrap_expand(points, multi, nboot, seed, chain0, ctx=None):
    ctx = _ctx(ctx)
    points = f64(points)
    N, n = points.shape
    out = np.empty(nboot)
    ctx.check(ctx.lib.b2n_bootstrap_expand(ctx.h, ptr(points), N, n, int(bool(multi)), nboot, seed,
                                           chain0, ptr(out)))
    return out


# ---- RadFriends / SupFriends (include/b200nest.h, b2n_friends_*) ---------------------------------
def friends_update(points, kind, am_prev=None, use_clustering=True, nboot=0, seed=0, chain0=0, ctx=None):
    """RadFriends.update / SupFriends.update (bounding.py:874-958 / 1142-1226).  kind: 'balls' | 'cubes'.
    Returns dict(cov, am, axes, axes_inv, logvol, radius, nclusters)."""
    ctx = _ctx(ctx)
    points = f64(points)
    N, n = points.shape
    o = dict(cov=np.empty((n, n)), am=np.empty((n, n)), axes=np.empty((n, n)), axes_inv=np.empty((n, n)))
    lv, rad, ncl = C.c_double(0.0), C.c_double(0.0), C.c_int32(0)
    amp = f64(am_prev) if (use_clustering and am_prev is not None) else None
    ctx.check(ctx.lib.b2n_friends_update(ctx.h, ptr(points), N, n, {'balls': 0, 'cubes': 1}[kind],
                                         int(bool(use_clustering and amp is not None)), ptr(amp), int(nboot), int(seed),
                                         int(chain0), ptr(o['cov']), ptr(o['am']), ptr(o['axes']), ptr(o['axes_inv']),
                                         C.addressof(lv), C.addressof(rad), C.addressof(ncl)))
    o.update(logvol=lv.value, radius=rad.value, nclusters=ncl.value)
    return o


def friends_set(kind, ctrs, axes, axes_inv, ctx=None, key=None):
    """Make (ctrs, axes, axes_inv) the resident friends bound of the ctx."""
    ctx = _ctx(ctx)
    ctrs, axes, axes_inv = f64(ctrs), f64(axes), f64(axes_inv)
    N, n = ctrs.shape
    ctx.friends_key = None
    ctx.check(ctx.lib.b2n_friends_set(ctx.h, {'balls': 0, 'cubes': 1}[kind], ptr(ctrs), N, n, ptr(axes), ptr(axes_inv)))
    ctx.friends_key = key


def friends_overlap(x, ctx=None):
    """q (M,) int32: number of balls / cubes of the resident friends bound containing each row of x."""
    ctx = _ctx(ctx)
    x = f64(np.atleast_2d(x))
    q = np.empty(len(x), dtype=np.int32)
    ctx.check(ctx.lib.b2n_friends_overlap(ctx.h, ptr(x), len(x), x.shape[1], ptr(q)))
    return q


def friends_unif_batch(model, nchain, ndim, loglstar, seed, chain0=0, dimflags=None, ctx=None, draw_only=False,
                       mixture=False):
    """UniformBoundSampler.sample x nchain on the resident friends bound; draw_only: Bound.samples(nchain)."""
    ctx = _ctx(ctx)
    a, keep, Q, n = _chain_args(model, None, ndim, loglstar, 1.0, seed, chain0, None, dimflags, Q=int(nchain), ndim=int(ndim))
    if draw_only:
        a.reserved = 3 if mixture else 1
    o = dict(u=np.empty((Q, n)), v=np.empty((Q, n)), logl=np.empty(Q), ncall=np.empty(Q, dtype=np.int32),
             nprop=np.empty(Q, dtype=np.int32), flags=np.empty(Q, dtype=np.uint32))
    ctx.check(ctx.lib.b2n_friends_unif_batch(ctx.h, C.byref(a), ptr(o['u']), ptr(o['v']), ptr(o['logl']), ptr(o['ncall']),
                                             ptr(o['nprop']), ptr(o['flags'])))
    if not draw_only and (o['flags'] & 0x80000000).any():
        raise NotImplementedError("uniform sampling did not find a point (bound draw limit)")
    return o


def bound_set(axes, ctrs=None, ams=None, logvols=None, ctx=None, key=None):
    """Make K ellipsoids resident for the proposal kernels (axes: (K, nc, nc)).
    A ctx holds ONE resident bound; `key` (the uploading bound's version token, None = anonymous) is
    recorded on the Context so that every user of the ctx can tell whether its bound is still the
    resident one (``ensure_resident``)."""
    ctx = _ctx(ctx)
    ctx.resident_key = None
    axes = f64(axes)
    if axes.ndim == 2:
        axes = axes[None]
    K, nc, _ = axes.shape
    if ctrs is not None:
        ctrs, ams, logvols = f64(ctrs).reshape(K, nc), f64(ams).reshape(K, nc, nc), f64(logvols).reshape(K)
    ctx.check(ctx.lib.b2n_bound_set(ctx.h, K, nc, ptr(ctrs), ptr(ams), ptr(axes), ptr(logvols)))
    ctx.resident_key = key


def ensure_resident(bound, ctx=None):
    """Upload `bound` (a B200 bound) unless it already is the resident bound of the ctx."""
    ctx = _ctx(ctx if ctx is not None else getattr(bound, 'ctx', None))
    if ctx.resident_key is None or ctx.resident_key != bound.version:
        bound.make_resident()


def _chain_args(model, u0, ncdim, loglstar, scale, seed, chain0, ell, dimflags, Q=None, ndim=None):
    a = ChainArgs()
    keep = []
    if u0 is not None:
        if not hasattr(u0, 'data_ptr'):          # numpy (host mode); torch tensors pass through
            u0 = f64(np.atleast_2d(u0))
        Q, ndim = int(u0.shape[0]), int(u0.shape[1])
        keep.append(u0)
    a.nchain, a.ndim, a.ncdim, a.model_id = Q, ndim, (ncdim or ndim), model
    a.u0 = ptr(u0)
    if ell is not None:
        ell = np.ascontiguousarray(ell, dtype=np.int32)
        keep.append(ell)
    a.ell = ptr(ell)
    if dimflags is not None:
        dimflags = np.ascontiguousarray(dimflags, dtype=np.uint8)
        keep.append(dimflags)
    a.dimflags = ptr(dimflags)
    a.loglstar, a.scale, a.seed, a.chain0 = float(loglstar), float(scale), int(seed), int(chain0)
    return a, keep, Q, ndim


def dimflags_from(ndim, periodic=None, reflective=None):
    """B2N_DIM_* flags from dynesty's periodic / reflective index lists."""
    if periodic is None and reflective is None:
        return None
    f = np.zeros(ndim, dtype=np.uint8)
    if periodic is not None:
        f[np.asarray(periodic, dtype=int)] |= _lib.DIM_PERIODIC
    if reflective is not None:
        f[np.asarray(reflective, dtype=int)] |= _lib.DIM_REFLECTIVE
    return f


class _gather:
    """Context manager for the fused multi-GPU gather (include/b200nest.h, peer section):
    `peer = (row0, total_rows)` makes the chains of the call rows [row0, row0 + Q) of a
    total_rows-chain fill whose outputs come back COMPLETE (all ranks' rows)."""

    def __init__(self, ctx, peer):
        self.ctx, self.peer = ctx, peer

    def __enter__(self):
        if self.peer is not None:
            self.ctx.peer_rows(self.peer[0], self.peer[1])

    def __exit__(self, *exc):
        if self.peer is not None:
            self.ctx.peer_rows(0, 0)
        return False


_NO_OUT = {}          # out=ops.NO_OUT: gather mode, device-pointer callers that read the window
NO_OUT = _NO_OUT


def rwalk_batch(model, u0, loglstar, scale, walks, seed, chain0=0, ncdim=None, ell=None,
                dimflags=None, ctx=None, out=None, peer=None, start_rows=None):
    """RWalkSampler.sample for every row of u0 (internal_samplers.py:505-561).
    `out`: optional dict of preallocated buffers (numpy, or torch tensors on the ctx device
    when the ctx is in device-pointer mode) with keys u, v, logl, n_accept, n_reject, ncall.
    `peer=(row0, total)`: fused multi-GPU gather, outputs have `total` rows.
    `start_rows`: int32 indices -- `u0` is then the whole live set and chain q starts from row start_rows[q]
    (b2n_set_start_rows: the gather of Sampler._fill_queue done by the kernel)."""
    ctx = _ctx(ctx)
    a, keep, Q, n = _chain_args(model, u0, ncdim, loglstar, scale, seed, chain0, ell, dimflags)
    if start_rows is not None:
        if not hasattr(start_rows, 'data_ptr'):
            start_rows = np.ascontiguousarray(start_rows, dtype=np.int32)
        keep.append(start_rows)
        a.nchain = int(start_rows.shape[0])
        ctx.set_start_rows(ptr(start_rows), Q)          # Q rows of u0 = the live set
        Q = a.nchain
    R = Q if peer is None else int(peer[1])
    o = out if out is not None else dict(
        u=np.empty((R, n)), v=np.empty((R, n)), logl=np.empty(R),
        n_accept=np.empty(R, dtype=np.int32), n_reject=np.empty(R, dtype=np.int32),
        ncall=np.empty(R, dtype=np.int32))
    g = o.get
    with _gather(ctx, peer):
        ctx.check(ctx.lib.b2n_rwalk_batch(ctx.h, C.byref(a), int(walks), ptr(g('u')), ptr(g('v')),
                                          ptr(g('logl')), ptr(g('n_accept')), ptr(g('n_reject')),
                                          ptr(g('ncall'))))
    return o


def _slice_batch(fn, model, u0, loglstar, scale, slices, seed, chain0, doubling, ell, ctx, peer=None):
    ctx = _ctx(ctx)
    a, keep, Q, n = _chain_args(model, u0, None, loglstar, scale, seed, chain0, ell, None)
    R = Q if peer is None else int(peer[1])
    o = dict(u=np.empty((R, n)), v=np.empty((R, n)), logl=np.empty(R),
             n_expand=np.empty(R, dtype=np.int32), n_contract=np.empty(R, dtype=np.int32),
             ncall=np.empty(R, dtype=np.int32), flags=np.empty(R, dtype=np.uint32))
    with _gather(ctx, peer):
        ctx.check(getattr(ctx.lib, fn)(ctx.h, C.byref(a), int(slices), int(bool(doubling)), ptr(o['u']),
                                       ptr(o['v']), ptr(o['logl']), ptr(o['n_expand']), ptr(o['n_contract']),
                                       ptr(o['ncall']), ptr(o['flags'])))
    return o


def rslice_batch(model, u0, loglstar, scale, slices, seed, chain0=0, doubling=False, ell=None, ctx=None,
                 peer=None):
    """RSliceSampler.sample per row of u0 (internal_samplers.py:745-855)."""
    return _slice_batch('b2n_rslice_batch', model, u0, loglstar, scale, slices, seed, chain0, doubling, ell, ctx,
                        peer)


def slice_batch(model, u0, loglstar, scale, slices, seed, chain0=0, doubling=False, ell=None, ctx=None,
                peer=None):
    """SliceSampler.sample per row of u0 (internal_samplers.py:593-709)."""
    return _slice_batch('b2n_slice_batch', model, u0, loglstar, scale, slices, seed, chain0, doubling, ell, ctx,
                        peer)


def unif_batch(model, nchain, ndim, loglstar, seed, chain0=0, ncdim=None, dimflags=None, ctx=None,
               draw_only=False, mixture=False, peer=None):
    """UniformBoundSampler.sample x nchain on the resident bound (internal_samplers.py:243-340).
    draw_only=True: just Bound.samples(nchain) (no cube test / likelihood)."""
    ctx = _ctx(ctx)
    a, keep, Q, n = _chain_args(model, None, ncdim, loglstar, 1.0, seed, chain0, None, dimflags,
                                Q=int(nchain), ndim=int(ndim))
    if draw_only:
        a.reserved = 3 if mixture else 1      # mixture: no 1/q test, q returned in 'ncall'
    R = Q if peer is None else int(peer[1])
    o = dict(u=np.empty((R, n)), v=np.empty((R, n)), logl=np.empty(R), ncall=np.empty(R, dtype=np.int32),
             nprop=np.empty(R, dtype=np.int32), flags=np.empty(R, dtype=np.uint32))
    with _gather(ctx, peer):
        ctx.check(ctx.lib.b2n_unif_batch(ctx.h, C.byref(a), ptr(o['u']), ptr(o['v']), ptr(o['logl']),
                                         ptr(o['ncall']), ptr(o['nprop']), ptr(o['flags'])))
    return o


def unitcube_batch(model, nchain, ndim, loglstar, seed, chain0=0, ctx=None, peer=None):
    """UnitCubeSampler.sample x nchain (internal_samplers.py:343-441): prior draws until logl > loglstar."""
    ctx = _ctx(ctx)
    a, keep, Q, n = _chain_args(model, None, None, loglstar, 1.0, seed, chain0, None, None, Q=int(nchain), ndim=int(ndim))
    R = Q if peer is None else int(peer[1])
    o = dict(u=np.empty((R, n)), v=np.empty((R, n)), logl=np.empty(R), ncall=np.empty(R, dtype=np.int32))
    with _gather(ctx, peer):
        ctx.check(ctx.lib.b2n_unitcube_batch(ctx.h, C.byref(a), ptr(o['u']), ptr(o['v']), ptr(o['logl']),
                                             ptr(o['ncall']), None))
    return o


# ---- device-resident nested-sampling rounds (include/b200nest.h, b2n_ns_*) ----------------------
def ns_create(model, nlive, ndim, batch, sampler, steps, seed, chain0=0, ncdim=None, strict_contains=True,
              facc=0.5, dlogz=0.01, maxiter=None, maxcall=None, update_interval=1 << 62, dimflags=None,
              dead_capacity=None, ctx=None, unit_cube_phase=False, first_min_ncall=0, first_min_eff=100., it0=0,
              logl_max=None):
    """Allocate the device state of a batched-replacement run (sampler: 0 rwalk, 1 rslice, 2 slice, 3 unif).
    unit_cube_phase: start with rounds that draw from the prior until the first bound is due
    (need_bound = 4 once ncall >= first_min_ncall and 100 (it0 + it) / ncall < first_min_eff)."""
    ctx = _ctx(ctx)
    c = _lib.NsConfig()
    c.nlive, c.ndim, c.ncdim, c.batch = int(nlive), int(ndim), int(ncdim or ndim), int(batch)
    c.sampler, c.steps, c.model_id, c.strict_contains = int(sampler), int(steps), int(model), int(bool(strict_contains))
    c.facc, c.dlogz = float(facc), float(dlogz)
    big = (1 << 62)
    c.maxiter = int(maxiter) if maxiter is not None else big
    c.maxcall = int(maxcall) if maxcall is not None else big
    c.update_interval, c.seed, c.chain0 = int(update_interval), int(seed), int(chain0)
    if dimflags is not None:
        dimflags = np.ascontiguousarray(dimflags, dtype=np.uint8)
    c.dimflags = ptr(dimflags)
    c.unit_cube_phase, c.first_min_ncall, c.first_min_eff, c.it0 = int(bool(unit_cube_phase)), int(first_min_ncall), \
        float(first_min_eff), int(it0)
    c.use_logl_max, c.logl_max = (0, 0.0) if logl_max is None else (1, float(logl_max))
    cap = int(dead_capacity) if dead_capacity is not None else 64 * int(nlive)
    ctx.check(ctx.lib.b2n_ns_create(ctx.h, C.byref(c), cap))


def ns_set_state(live_u, live_v, live_logl, logvol, logz, loglstar, ncall, scale, ctx=None):
    ctx = _ctx(ctx)
    live_u, live_v, live_logl = f64(live_u), f64(live_v), f64(live_logl)
    ctx.check(ctx.lib.b2n_ns_set_state(ctx.h, ptr(live_u), ptr(live_v), ptr(live_logl), float(logvol), float(logz),
                                       float(loglstar), 0, int(ncall), float(scale)))


def _ns_status(st):
    return {k: getattr(st, k) for k, _ in st._fields_}


def ns_run(max_rounds, check_every=0, ctx=None):
    """Enqueue up to max_rounds rounds; returns the status dict (it, ncall, rounds, logz, logvol, loglstar,
    lmax, delta_logz, scale, done, need_bound, doubling, error)."""
    ctx = _ctx(ctx)
    st = _lib.NsStatus()
    ctx.check(ctx.lib.b2n_ns_run(ctx.h, int(max_rounds), int(check_every), C.byref(st)))
    return _ns_status(st)


def ns_status(ctx=None):
    ctx = _ctx(ctx)
    st = _lib.NsStatus()
    ctx.check(ctx.lib.b2n_ns_status_get(ctx.h, C.byref(st)))
    return _ns_status(st)


def ns_set_counters(rounds, ncall_last_update, doubling, ctx=None):
    """Counters of a restored run (round index, calls at the last bound update, slice-doubling switch)."""
    ctx = _ctx(ctx)
    ctx.check(ctx.lib.b2n_ns_set_counters(ctx.h, int(rounds), int(ncall_last_update), int(bool(doubling))))


def ns_bound_updated(ctx=None):
    ctx = _ctx(ctx)
    ctx.check(ctx.lib.b2n_ns_bound_updated(ctx.h))


_ns_bound_serial = [0]


def ns_update_bound(multi, enlarge=1.0, ctx=None):
    """Sampler.update_bound on the device (b2n_ns_update_bound): fit the bound to the run's live points in HBM,
    enlarge, make resident.  Returns (nells, logvol, warn)."""
    ctx = _ctx(ctx)
    nells, warn, lv = C.c_int32(0), C.c_uint32(0), C.c_double(0.0)
    ctx.resident_key = None
    ctx.check(ctx.lib.b2n_ns_update_bound(ctx.h, int(bool(multi)), float(enlarge), C.addressof(nells), C.addressof(lv),
                                          C.addressof(warn)))
    _ns_bound_serial[0] += 1
    ctx.resident_key = ('ns', ctx.serial, _ns_bound_serial[0])     # no host bound object owns these ellipsoids
    return nells.value, lv.value, warn.value


def ns_get_bound(nells, ncdim, ctx=None):
    """The bound the last ns_update_bound built: dict(ctrs, covs, ams, axes, axlens, logvols)."""
    ctx = _ctx(ctx)
    K, n = int(nells), int(ncdim)
    o = dict(ctrs=np.empty((K, n)), covs=np.empty((K, n, n)), ams=np.empty((K, n, n)), axes=np.empty((K, n, n)),
             axlens=np.empty((K, n)), logvols=np.empty(K))
    ctx.check(ctx.lib.b2n_ns_get_bound(ctx.h, K, ptr(o['ctrs']), ptr(o['covs']), ptr(o['ams']), ptr(o['axes']),
                                       ptr(o['axlens']), ptr(o['logvols'])))
    return o


_FRIENDS_KIND = {'balls': 0, 'cubes': 1}


def ns_update_friends(kind, enlarge=1.0, nboot=0, use_clustering=True, ctx=None):
    """RadFriends / SupFriends update on the device (b2n_ns_update_friends): fit to the run's live points in HBM under
    the run's previous metric, enlarge, make it the run's bound.  kind: 'balls' | 'cubes'.
    Returns (logvol, radius, nclusters)."""
    ctx = _ctx(ctx)
    lv, rad, ncl = C.c_double(0.0), C.c_double(0.0), C.c_int32(0)
    ctx.resident_key = None
    ctx.check(ctx.lib.b2n_ns_update_friends(ctx.h, _FRIENDS_KIND[kind], float(enlarge), int(nboot), int(bool(use_clustering)),
                                            C.addressof(lv), C.addressof(rad), C.addressof(ncl)))
    _ns_bound_serial[0] += 1
    ctx.resident_key = ('ns', ctx.serial, _ns_bound_serial[0])     # the run's common axes; no host object owns them
    return lv.value, rad.value, ncl.value


def ns_set_friends(kind, cov, am, axes, axes_inv, logvol, ctx=None):
    """Adopt a RadFriends / SupFriends bound built on the host as the run's bound (centres: the run's live set)."""
    ctx = _ctx(ctx)
    cov, am, axes, axes_inv = f64(cov), f64(am), f64(axes), f64(axes_inv)
    ctx.resident_key = None
    ctx.check(ctx.lib.b2n_ns_set_friends(ctx.h, _FRIENDS_KIND[kind], ptr(cov), ptr(am), ptr(axes), ptr(axes_inv),
                                         float(logvol)))
    _ns_bound_serial[0] += 1
    ctx.resident_key = ('ns', ctx.serial, _ns_bound_serial[0])


def ns_get_friends(ndim, ctx=None):
    """The friends bound the run holds: dict(cov, am, axes, axes_inv, logvol, radius, nclusters) (an adopted bound:
    radius nan, nclusters 0)."""
    ctx = _ctx(ctx)
    n = int(ndim)
    o = dict(cov=np.empty((n, n)), am=np.empty((n, n)), axes=np.empty((n, n)), axes_inv=np.empty((n, n)))
    lv, rad, ncl = C.c_double(0.0), C.c_double(0.0), C.c_int32(0)
    ctx.check(ctx.lib.b2n_ns_get_friends(ctx.h, ptr(o['cov']), ptr(o['am']), ptr(o['axes']), ptr(o['axes_inv']),
                                         C.addressof(lv), C.addressof(rad), C.addressof(ncl)))
    o.update(logvol=lv.value, radius=rad.value, nclusters=ncl.value)
    return o


def ns_reserve_dead(capacity, ctx=None):
    ctx = _ctx(ctx)
    ctx.check(ctx.lib.b2n_ns_reserve_dead(ctx.h, int(capacity)))


def ns_get_live(nlive, ndim, ctx=None, only_u=False):
    ctx = _ctx(ctx)
    u = np.empty((nlive, ndim))
    if only_u:          # what a bound update needs
        ctx.check(ctx.lib.b2n_ns_get_live(ctx.h, ptr(u), None, None))
        return u
    v, l = np.empty((nlive, ndim)), np.empty(nlive)
    ctx.check(ctx.lib.b2n_ns_get_live(ctx.h, ptr(u), ptr(v), ptr(l)))
    return u, v, l


def ns_get_dead(first, count, ndim, ctx=None, positions=True):
    """(u, v, logl, logvol, ncall) of dead points [first, first + count); positions=False skips the two
    (count, ndim) position arrays (zero-row placeholders) -- the evidence needs only the scalars."""
    ctx = _ctx(ctx)
    u, v = (np.empty((count, ndim)), np.empty((count, ndim))) if positions else (None, None)
    l, lv, nc = np.empty(count), np.empty(count), np.empty(count, dtype=np.int32)
    ctx.check(ctx.lib.b2n_ns_get_dead(ctx.h, int(first), int(count), ptr(u), ptr(v), ptr(l), ptr(lv), ptr(nc)))
    if not positions:
        u, v = np.empty((0, ndim)), np.empty((0, ndim))
    return u, v, l, lv, nc


def ns_destroy(ctx=None):
    ctx = _ctx(ctx)
    ctx.check(ctx.lib.b2n_ns_destroy(ctx.h))
