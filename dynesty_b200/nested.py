"""Host mirror of the reference ``Sampler``'s proposal dispatch, batched for the GPU.

What is mirrored (reference py/dynesty/sampler.py, same names / meaning):
  propose_live            :469-491   start point + axes (+ contains check, forced update)
  update_bound            :493-510   bound.update(...) + enlarge via scale_to_logvol
  update_bound_if_needed  :625-674   first-update / interval / forced logic
  _fill_queue             :676-717   queue_size proposals per fill, ONE kernel launch
  _new_point              :732-778   pop until logl > loglstar; tune when the queue drains;
                                     bound update check when the queue is empty
and the factory defaults of dynesty.py (:126-135 walks/slices, :169-211 enlarge/bootstrap,
:213-230 update interval, sampler.py:407-409 first update).

The surrounding nested-sampling bookkeeping (dead-point record, evidence integral) is the
reference's L2/L4 layer and out of scope as a subsystem; the minimum needed to turn the
hot path into a logZ (the BASELINE metric's second half) is restated compactly in
``_integrate`` (utils.py:1411-1467) and ``run_nested`` (sampler.py:1040-1212, 780-914).
On a machine that has dynesty installed the same bounds/samplers plug into
``dynesty.NestedSampler`` directly (see INTEGRATION.md); this driver exists because the GPU
box has no dynesty, and because it proposes/contains-checks a whole queue per call.
"""
import heapq
import math

import numpy as np

from . import bounding as B
from . import samplers as S

LOWL = -1e300


def _logaddexp(a, b):
    if a < b:
        a, b = b, a
    if b == -math.inf:
        return a
    return a + math.log1p(math.exp(b - a))


class Results(dict):
    __getattr__ = dict.__getitem__

    def summary(self):
        return ("niter: %d\nncall: %d\neff(%%): %6.3f\nlogz: %6.3f +/- %6.3f" %
                (self['niter'], self['ncall'], self['eff'], self['logz'][-1], self['logzerr'][-1]))

    def posterior_moments(self):
        w = np.exp(self['logwt'] - self['logz'][-1])
        w /= w.sum()
        mean = w @ self['samples']
        d = self['samples'] - mean
        return mean, (d * w[:, None]).T @ d


def _integrate(logl, logvol):
    """Trapezoid evidence / information integrals over the dead-point sequence
    (utils.py:1411-1467 compute_integrals, same quadrature)."""
    lpad = np.concatenate([[LOWL], logl])
    dlv = np.diff(logvol, prepend=0)
    logdvol = logvol - dlv + np.log1p(-np.exp(dlv))
    logdvol2 = logdvol + math.log(0.5)
    logwt = np.logaddexp(lpad[1:], lpad[:-1]) + logdvol2
    logz = np.logaddexp.accumulate(logwt)
    zmax = logz[-1]
    h1 = np.cumsum(np.exp(lpad[1:] - zmax + logdvol2) * lpad[1:] +
                   np.exp(lpad[:-1] - zmax + logdvol2) * lpad[:-1])
    h = h1 - zmax * np.exp(logz - zmax)
    dh = np.diff(h, prepend=0)
    logzvar = np.abs(np.cumsum(dh * (-dlv)))
    return logwt, logz, logzvar, h


class NestedSampler:
    """Static nested sampler whose bound construction and proposal chains run on the GPU.

    Parameters follow dynesty.NestedSampler (dynesty.py:584-614); `model` is a
    ``DeviceModel`` instead of the (loglikelihood, prior_transform) callables.
    `comm`: optional ``dynesty_b200.dist.Comm`` -- chains of a queue fill are sharded over
    the ranks and all-gathered (NCCL), every rank keeps the identical host state.
    """

    def __init__(self, model, nlive=500, bound='multi', sample='auto', ncdim=None, walks=None, slices=None,
                 facc=0.5, enlarge=None, bootstrap=None, update_interval=None, first_update=None,
                 queue_size=None, periodic=None, reflective=None, seed=56432, ctx=None, comm=None, live_points=None,
                 live_init='device'):
        self.model = model
        self.ndim = n = model.ndim
        self.ncdim = ncdim or n
        self.nlive = int(nlive)
        self.rstate = np.random.default_rng(seed)
        self.seed = int(seed)
        self.ctx = ctx
        self.comm = comm
        # -- inner sampler (dynesty.py:126-166)
        if sample == 'auto':
            sample = 'unif' if n < 10 else ('rwalk' if n <= 20 else 'rslice')
        kw = dict(model=model, ndim=n, ncdim=self.ncdim, periodic=periodic, reflective=reflective, facc=facc,
                  ctx=ctx)
        if isinstance(sample, str):
            self.sample_name = sample
            if sample == 'rwalk':
                sample = S.B200RWalkSampler(walks=walks or n + 20, **kw)
            elif sample == 'rslice':
                sample = S.B200RSliceSampler(slices=slices or 3 + n, **kw)
            elif sample == 'slice':
                sample = S.B200SliceSampler(slices=slices or 3, **kw)
            elif sample == 'unif':
                sample = S.B200UniformSampler(**kw)
            else:
                raise ValueError("Unknown sampling method: '%s'" % sample)
        else:
            self.sample_name = type(sample).__name__
        if self.ncdim != n and isinstance(sample, S._B200SliceBase):
            raise ValueError('ncdim unsupported for slice sampling')          # dynesty.py:505-507
        self.internal_sampler_next = sample
        # -- bound (sampler.py:28-53)
        if bound == 'multi':
            bound = B.B200MultiEllipsoid(self.ncdim, ctx=ctx)
        elif bound == 'single':
            bound = B.B200Ellipsoid(self.ncdim, ctx=ctx)
        elif bound in ('balls', 'cubes'):
            if self.ncdim != n:
                raise ValueError('ncdim unsupported for the friends bounds')
            bound = (B.B200RadFriends if bound == 'balls' else B.B200SupFriends)(n, ctx=ctx)
        elif bound == 'none':
            bound = None
        elif isinstance(bound, str):
            raise ValueError("Unknown bounding method: %s (B200 path: none/single/multi/balls/cubes)" % bound)
        self.bound_next = bound
        self.bound = None
        self.unit_cube_sampling = True
        # -- enlarge / bootstrap defaults (dynesty.py:169-211)
        is_unif = isinstance(sample, S.B200UniformSampler)
        if enlarge is not None and bootstrap is None:
            bootstrap = 0
        elif enlarge is None and bootstrap is not None:
            enlarge = 1
        elif enlarge is None and bootstrap is None:
            enlarge, bootstrap = (1, 5) if is_unif else (1.25, 0)
        elif not (bootstrap == 0 or enlarge == 1):
            raise ValueError('Enlarge and bootstrap together do not make sense unless '
                             'bootstrap=0 or enlarge = 1')
        self.bound_enlarge, self.bound_bootstrap = float(enlarge), int(bootstrap)
        # -- update interval in calls (dynesty.py:213-240, 646-649)
        if update_interval is None:
            ratio = sample.update_bound_interval_ratio
        elif isinstance(update_interval, float):
            ratio = update_interval
        else:
            ratio = int(update_interval) / self.nlive
        self.bound_update_interval = int(max(round(ratio * self.nlive), 1))
        fu = first_update or {}
        self.first_bound_update_ncall = fu.get('min_ncall', 2 * self.nlive)    # sampler.py:407-409
        self.first_bound_update_eff = fu.get('min_eff', 10.)
        self.logl_first_update = None
        self.ncall_at_last_update = 0
        self.queue_size = int(queue_size or self.nlive)
        if comm is not None and self.queue_size % comm.world:
            self.queue_size += comm.world - self.queue_size % comm.world
        # -- live points (sampler.py:56-262, evaluated in one launch)
        if live_points is not None:         # (u, v, logl) supplied by the caller (dynesty.py:600 `live_points`)
            self.live_u, self.live_v, self.live_logl = (np.array(a, dtype=float) for a in live_points)
        elif live_init == 'device':
            # _initialize_live_points (sampler.py:56-262) on the device: nlive prior draws + transform + likelihood in
            # ONE launch (b2n_unitcube_batch at threshold -inf: a draw whose logl is -inf is redrawn, the reference's
            # "keep the finite ones" rule :167-200 for a queue of one).  Chain ids 2^61 + i: disjoint from the run's.
            from . import ops
            o = ops.unitcube_batch(model.model_id(ctx), self.nlive, n, -np.inf, self.seed, chain0=1 << 61, ctx=ctx)
            self.live_u, self.live_v, self.live_logl = o['u'], o['v'], o['logl']
            self.init_ncall = int(o['ncall'].sum())
        else:
            self.live_u = self.rstate.random((self.nlive, n))
            self.live_v, self.live_logl = model.evaluate(self.live_u, ctx=ctx)
        self.it = 1
        self.ncall = getattr(self, 'init_ncall', self.nlive)
        self.eff = 0.
        self.nbound = 1
        self.chain_counter = 0
        self.scale_history = []
        self.nbatches = 0
        self.n_proposals = 0
        self.bound_history = []           # (ncall, nells, logvol) per update
        self._q = None
        self._qpos = 0

    # ------------------------------------------------------------------ save / restore (utils.py:2321-2355)
    def __getstate__(self):
        d = self.__dict__.copy()
        d['ctx'] = d['comm'] = None                  # device handles are per process
        return d

    def save(self, fname):
        """Pickle the sampler (the reference's ``save_sampler``): with loop='device' the pickle carries the
        snapshot of the device-resident run taken at the last consistent point (``_dev_snap``)."""
        import os
        import pickle
        tmp = fname + '.tmp'
        with open(tmp, 'wb') as f:
            pickle.dump(self, f, protocol=pickle.HIGHEST_PROTOCOL)
        os.replace(tmp, fname)                        # atomic, like utils.py:2343-2352

    @classmethod
    def restore(cls, fname, ctx=None):
        """``restore_sampler``: continue with ``run_nested(resume=True)``."""
        import pickle
        with open(fname, 'rb') as f:
            ns = pickle.load(f)
        ns.ctx = ctx
        for o in (ns.bound, ns.bound_next, getattr(ns, 'internal_sampler', None), ns.internal_sampler_next):
            if o is not None and hasattr(o, '_ctx'):
                o._ctx = ctx
            if o is not None and hasattr(o, '_m'):
                o._m._ctx = ctx
        return ns

    # ------------------------------------------------------------------ bounds
    def _ensure_resident(self):
        from . import ops, _lib
        c = self.ctx if self.ctx is not None else _lib.default_context()
        if c.resident_key is None or c.resident_key != self.bound.version:
            self.bound.make_resident(c)

    def update_bound(self, subset=slice(None)):
        """sampler.py:493-510."""
        if getattr(self.bound, 'need_centers', False):
            self.bound.ctrs = self.live_u
        if self.comm is not None and isinstance(self.bound, B.B200Ellipsoid) and self.bound_bootstrap == 0 and \
                isinstance(subset, slice) and getattr(self, 'shard_bound_update', True):
            # the rows of the live set are dealt over the ranks: each reduces its share, all-reduce of the moments
            lo, hi = (self.nlive * self.comm.rank) // self.comm.world, (self.nlive * (self.comm.rank + 1)) // self.comm.world
            self.bound.update_sharded(self.live_u[lo:hi, :self.ncdim], self.comm)
            if self.bound_enlarge != 1.:
                self.bound.scale_to_logvol(self.bound.logvol + math.log(self.bound_enlarge))
            return
        self.bound.update(self.live_u[subset, :self.ncdim], rstate=self.rstate, bootstrap=self.bound_bootstrap)
        if self.bound_enlarge != 1.:
            self.bound.scale_to_logvol(self.bound.logvol + math.log(self.bound_enlarge))

    def update_bound_if_needed(self, loglstar, ncall=None, force=False):
        """sampler.py:625-674."""
        if self.bound_next is None:
            return
        ncall = self.ncall if ncall is None else ncall
        call_check_first = ncall >= self.first_bound_update_ncall
        call_check = ncall >= self.bound_update_interval + self.ncall_at_last_update
        eff_check = self.eff < self.first_bound_update_eff
        ucs = self.unit_cube_sampling
        if ((ucs and eff_check and call_check_first) or (not ucs and call_check) or
                (ucs and self.logl_first_update is not None and loglstar > self.logl_first_update) or force):
            subset = (self.live_logl > loglstar) if loglstar == LOWL else slice(None)
            if ucs:
                self.unit_cube_sampling = False
                self.logl_first_update = loglstar
                self.bound = self.bound_next
                self.internal_sampler = self.internal_sampler_next
            self.update_bound(subset)
            self.nbound += 1
            self.ncall_at_last_update = ncall
            self.bound_history.append((ncall, getattr(self.bound, 'nells', 1), float(self.bound.logvol)))

    # ------------------------------------------------------------------ proposals
    def propose_live(self, loglstar, size):
        """sampler.py:469-491 for a whole queue: start rows + ellipsoid indices."""
        idx = np.nonzero(self.live_logl > loglstar)[0]
        if len(idx) == 0:
            raise RuntimeError('No live points are above loglstar. Do you have a likelihood plateau ?')
        starts = idx[self.rstate.integers(len(idx), size=size)]
        uniq = np.unique(starts)
        if not self.bound.contains_many(self.live_u[uniq, :self.ncdim]).all():
            self.update_bound_if_needed(-np.inf, force=True)
            if not self.bound.contains_many(self.live_u[uniq, :self.ncdim]).all():
                raise RuntimeError('Update of the ellipsoid failed')
        ell = self.bound.random_ells(self.rstate, size)
        return starts, ell

    def _run_sharded(self, fn, Q, fused=True):
        """Run chains [lo, hi) of a Q-chain fill on this rank and gather all ranks' chains:
        inside the kernel over NVLink peer windows when the Comm has them (dist.attach_peer),
        else with one all-gather per output array."""
        if self.comm is None:
            return fn(0, Q, None)
        lo, hi = self.comm.shard(Q)
        if fused and self.comm.peer_ctx is not None:
            return fn(lo, hi, (lo, Q))
        return self.comm.allgather(fn(lo, hi, None), Q)

    def _fill_queue(self, loglstar):
        """sampler.py:676-717: one launch for `queue_size` proposals."""
        Q = self.queue_size
        c0 = self.chain_counter
        self.chain_counter += Q
        if not self.unit_cube_sampling and getattr(self.bound, 'need_centers', False):
            self.bound.ctrs = self.live_u                                  # sampler.py:479-482
        if self.unit_cube_sampling:
            # UnitCubeSampler (internal_samplers.py:343-441): u ~ U(0,1)^n, one call each
            u = self.rstate.random((Q, self.ndim))

            def fn(lo, hi, peer):
                v, l = self.model.evaluate(u[lo:hi], ctx=self.ctx)
                return dict(u=u[lo:hi], v=v, logl=l, ncall=np.ones(hi - lo, dtype=np.int32))
            q = self._run_sharded(fn, Q, fused=False)
        else:
            smp = self.internal_sampler
            if isinstance(smp, S.B200UniformSampler):
                def fn(lo, hi, peer):
                    return smp.run_batch(loglstar, hi - lo, self.bound, self.seed, chain0=c0 + lo, ncdim=self.ncdim,
                                         peer=peer)
            else:
                starts, ell = self.propose_live(loglstar, Q)
                pts = np.take(self.live_u, starts, axis=0, mode='clip')       # (valid rows by construction)
                # device copy of the bound follows the host object (one resident bound per ctx, tracked on the
                # Context: ops.ensure_resident)
                self._ensure_resident()

                def fn(lo, hi, peer):
                    return smp.run_batch(loglstar, pts[lo:hi], ell[lo:hi], self.seed, chain0=c0 + lo, peer=peer)
            q = self._run_sharded(fn, Q)
        self.nbatches += 1
        self.n_proposals += int(q['ncall'].sum())
        self._q = q
        self._ql = q['logl'].tolist()
        self._qn = q['ncall'].tolist()
        self._qpos = 0

    def _queue_drained(self, loglstar):
        """The part of _new_point that runs when the last queue item has been popped
        (sampler.py:757-772): tune with update=True, then the bound-update check."""
        q = self._q
        if not self.unit_cube_sampling:
            smp = self.internal_sampler
            if 'n_accept' in q:
                smp.tune({'accept': int(q['n_accept'].sum()), 'reject': int(q['n_reject'].sum()),
                          'scale': smp.scale}, update=True)
            elif 'n_expand' in q:
                warned = bool((q['flags'] & 2).any())
                smp.tune({'n_expand': int(q['n_expand'].sum()), 'n_contract': int(q['n_contract'].sum()),
                          'expansion_warning_set': warned}, update=True)
            self.scale_history.append((self.ncall, smp.scale))
        self.update_bound_if_needed(loglstar, ncall=self.ncall)

    # ------------------------------------------------------------------ device-resident rounds
    def _device_bound_ok(self):
        """The bound can be rebuilt without leaving the device (b2n_ns_update_bound): one of the library's own
        ellipsoid bounds and no bootstrap expansion."""
        b = self.bound_next
        return type(b) in (B.B200MultiEllipsoid, B.B200Ellipsoid) and self.bound_bootstrap == 0 and \
            getattr(self, 'device_bound', True)

    def _pull_device_bound(self, nells):
        """Host bound object <- the bound the device built (results, checkpoints, plotting read self.bound)."""
        from . import ops
        o = ops.ns_get_bound(nells, self.ncdim, ctx=self.ctx)
        m = self.bound._m if isinstance(self.bound, B.B200Ellipsoid) else self.bound
        m.nells = nells
        m.ctrs, m.covs, m.ams = o['ctrs'], o['covs'], o['ams']
        m.axes_all, m.axlens_all, m.logvol_ells = o['axes'], o['axlens'], o['logvols']
        m._refresh_logvol()
        c = self.ctx if self.ctx is not None else m.ctx
        c.resident_key = m.version                     # these very ellipsoids ARE the resident bound

    def _pull_device_friends(self, ctrs):
        """Host RadFriends / SupFriends object <- the bound the device rounds hold; its centres are `ctrs` (the live
        set the device bound was used with).  The ctx's resident axes stay anonymous: no host object claims them."""
        from . import ops
        o = ops.ns_get_friends(self.ndim, ctx=self.ctx)
        b = self.bound
        b.cov, b.am, b.axes, b.axes_inv, b.logvol = o['cov'], o['am'], o['axes'], o['axes_inv'], float(o['logvol'])
        if o['nclusters'] > 0:                         # (an adopted bound reports none: the object's own values stand)
            b.radius, b.nclusters = o['radius'], o['nclusters']
        b.ctrs = ctrs
        b.version = next(B._version)

    def _device_rounds(self, logz, logvol, loglstar, dlogz, maxiter, maxcall, batch, checkpoint_file=None,
                       checkpoint_every=0.0, snap=None, on_checkpoint=None, keep_samples=True, logl_max=None):
        """Run (or continue) with ``b2n_ns_run`` (include/b200nest.h): K-worst replacement rounds paced on the
        device -- first with prior draws (the phase before the first bound, sampler.py:407-409), then with the
        inner sampler against the resident bound.  The host only reacts to the device's flags: (re)build the bound
        (update_bound, sampler.py:493-510 -- on the device when ``_device_bound_ok``), grow the dead buffer, and
        collect the dead points at the end.  With a RadFriends / SupFriends bound every update runs on the device
        (``b2n_ns_update_friends``, bootstrap included) and a bound built beforehand is adopted as it is."""
        from . import ops
        import time
        n, N = self.ndim, self.nlive
        smp = self.internal_sampler_next
        kind = (0 if isinstance(smp, S.B200RWalkSampler) else 1 if isinstance(smp, S.B200RSliceSampler) else
                2 if isinstance(smp, S.B200SliceSampler) else 3)             # 3: uniform sampler (no chains to tune)
        steps = 1 if kind == 3 else smp.sampler_kwargs['walks' if kind == 0 else 'slices']
        # default batch: rwalk chains use a proposal shape estimated from the live points and mix slowly along
        # under-estimated directions; the resulting logZ bias grows with the fraction of the live set replaced
        # per round (DESIGN.md 9.4): nlive/40 reproduces the reference's serial result.  Slice chains
        # decorrelate: nlive/10.
        K = int(batch or max(1, N // (40 if kind == 0 else 10)))
        self.batch = K
        prev = [np.empty((0, n)), np.empty((0, n)), np.empty(0), np.empty(0), np.empty(0, dtype=np.int32)]
        chain_base = self.chain_counter
        it0_orig = it0 = self.it         # iterations before the device phase (enters the efficiency test)
        if snap is not None:             # resume: rows that died before the snapshot, scalars of the run
            prev = [snap['dead'][k] for k in range(5)]
            self.live_u, self.live_v, self.live_logl = snap['live']
            logvol, logz, loglstar = snap['logvol'], snap['logz'], snap['loglstar']
            self.ncall, smp.scale, chain_base = snap['ncall'], snap['scale'], snap['chain_base']
            maxiter = maxiter - len(prev[2]) if maxiter < (1 << 61) else maxiter
            it0_orig = snap['it0']
            it0 = it0_orig + len(prev[2])
        no_bound = self.bound_next is None
        friends = isinstance(self.bound_next, B._B200Friends)
        if friends and self.bound_bootstrap > 255:
            raise ValueError("loop='device' with the friends bounds: bootstrap <= 255 (one chain id per realisation)")
        multi = not isinstance(self.bound_next, B.B200Ellipsoid)
        ops.ns_create(self.model.model_id(self.ctx), N, n, K, kind, steps, self.seed, chain0=chain_base,
                      ncdim=self.ncdim, strict_contains=multi,
                      facc=getattr(smp, 'facc', 0.5), dlogz=dlogz if dlogz is not None else 0.0,
                      maxiter=maxiter if maxiter < (1 << 61) else None, maxcall=maxcall,
                      update_interval=self.bound_update_interval, dimflags=smp._flags(), ctx=self.ctx,
                      unit_cube_phase=self.unit_cube_sampling,
                      first_min_ncall=(1 << 62) if no_bound else self.first_bound_update_ncall,
                      first_min_eff=self.first_bound_update_eff, it0=it0, logl_max=logl_max)
        tm = dict(rounds_s=0.0, bound_s=0.0)
        self.device_timing = tm
        st = None
        try:
            ops.ns_set_state(self.live_u, self.live_v, self.live_logl, logvol, logz, loglstar, self.ncall, smp.scale,
                             ctx=self.ctx)
            rounds0 = 0
            if snap is not None:
                rounds0 = snap['rounds']
                ops.ns_set_counters(snap['rounds'], snap['ncall_last_update'], snap['doubling'], ctx=self.ctx)
            if not self.unit_cube_sampling:
                if friends:                           # resume / dynamic batch: the bound built so far, centred on the live set
                    b = self.bound
                    ops.ns_set_friends(b.kind, b.cov, b.am, b.axes, b.axes_inv, b.logvol, ctx=self.ctx)
                else:
                    self._ensure_resident()
            cap, last_forced = 64 * N, -1
            ncall_start, rounds = self.ncall, rounds0
            t_ckpt, n_ckpt, saved_it = time.perf_counter(), 0, 0
            dev_nells = 0

            def checkpoint(st):
                """Snapshot at a consistent point (flags clear, bound current): live set, scalars, the rows that
                died since the last snapshot; then pickle the whole sampler (host phase results included)."""
                nonlocal saved_it, prev
                new = ops.ns_get_dead(saved_it, st['it'] - saved_it, n, ctx=self.ctx)
                prev = [np.concatenate([a, b]) for a, b in zip(prev, new)]
                saved_it = st['it']
                if dev_nells:
                    self._pull_device_bound(dev_nells)
                live = ops.ns_get_live(N, n, ctx=self.ctx)
                if friends:
                    self._pull_device_friends(live[0])
                self._dev_snap = dict(dead=prev, live=live, logvol=st['logvol'],
                                      logz=st['logz'], loglstar=st['loglstar'], ncall=st['ncall'], scale=st['scale'],
                                      rounds=st['rounds'], ncall_last_update=st['ncall_last_update'],
                                      doubling=st['doubling'], chain_base=chain_base, batch=K, it0=it0_orig)
                self.save(checkpoint_file)

            while True:
                done_r = rounds - rounds0
                if self.unit_cube_sampling:           # prior draws: ~100/eff calls per accepted point
                    per_round = max(1.0, (self.ncall - ncall_start) / done_r) if done_r else 2.0 * K
                    due = self.first_bound_update_ncall - self.ncall
                    want = int(min(64, max(1, math.ceil(due / per_round)))) if not no_bound else 256
                else:
                    per_round = max(1.0, (self.ncall - ncall_start) / done_r) if done_r else K * steps * (1 if kind == 0 else 6)
                    if kind == 3 and not done_r:
                        per_round = K * max(1.0, 100. / max(self.eff, 1.))        # uniform draws: ~1/eff calls each
                    due = self.ncall_at_last_update + self.bound_update_interval - self.ncall
                    want = int(min(4096, max(1, math.ceil(due / per_round))))
                t0 = time.perf_counter()
                st = ops.ns_run(want, 0, ctx=self.ctx)
                tm['rounds_s'] += time.perf_counter() - t0
                rounds, self.ncall = st['rounds'], st['ncall']
                self.eff = 100. * (it0 + st['it']) / max(self.ncall, 1)
                self.scale_history.append((self.ncall, st['scale']))
                if st['done']:
                    break
                if st['need_bound'] == 3:                               # dead-point buffer full
                    cap *= 2
                    ops.ns_reserve_dead(cap, ctx=self.ctx)
                elif st['need_bound']:
                    if st['need_bound'] == 2:                           # a start point outside the bound
                        if last_forced == rounds:
                            raise RuntimeError('Update of the ellipsoid failed')     # sampler.py:489
                        last_forced = rounds
                    t0 = time.perf_counter()
                    if st['need_bound'] == 4:                           # first bound (sampler.py:640-647)
                        self.unit_cube_sampling = False
                        self.logl_first_update = st['loglstar']
                        self.bound = self.bound_next
                        self.internal_sampler = self.internal_sampler_next
                        ncall_start, rounds0 = self.ncall, rounds      # calls per round change with the sampler
                    if friends:
                        lv, _, _ = ops.ns_update_friends(self.bound.kind, self.bound_enlarge, self.bound_bootstrap,
                                                         use_clustering=True, ctx=self.ctx)
                        nells = 1
                    elif self._device_bound_ok():
                        dev_nells, lv, warn = ops.ns_update_bound(multi, self.bound_enlarge, ctx=self.ctx)
                        nells = dev_nells
                    else:
                        self.live_u = ops.ns_get_live(N, n, ctx=self.ctx, only_u=True)
                        self.update_bound()
                        self._ensure_resident()
                        dev_nells, nells, lv = 0, getattr(self.bound, 'nells', 1), float(self.bound.logvol)
                    self.nbound += 1
                    self.ncall_at_last_update = self.ncall
                    self.bound_history.append((self.ncall, nells, lv))
                    ops.ns_bound_updated(ctx=self.ctx)
                    tm['bound_s'] += time.perf_counter() - t0
                    if checkpoint_file is not None and time.perf_counter() - t_ckpt >= checkpoint_every:
                        st = ops.ns_status(ctx=self.ctx)              # flags cleared, interval restarted
                        checkpoint(st)
                        t_ckpt, n_ckpt = time.perf_counter(), n_ckpt + 1
                        if on_checkpoint is not None:
                            on_checkpoint(n_ckpt)
            if not self.unit_cube_sampling:
                smp.scale = st['scale']
                if st['doubling']:
                    smp.sampler_kwargs['slice_doubling'] = True
                if dev_nells:
                    self._pull_device_bound(dev_nells)
            self.live_u, self.live_v, self.live_logl = ops.ns_get_live(N, n, ctx=self.ctx)
            if friends and not self.unit_cube_sampling:
                self._pull_device_friends(self.live_u)
            new = ops.ns_get_dead(saved_it, st['it'] - saved_it, n, ctx=self.ctx, positions=keep_samples)
            out = tuple(np.concatenate([a, b]) for a, b in zip(prev, new))
            self.chain_counter = chain_base + rounds * K
            self.nbatches += rounds - (snap['rounds'] if snap is not None else 0)
            self.n_proposals += self.ncall - ncall_start
            self.it = it0 + st['it']
            self.device_rounds = rounds
            self._dev_snap = None
            return out
        finally:
            ops.ns_destroy(ctx=self.ctx)            # also on errors: the device state never outlives the call

    # ------------------------------------------------------------------ main loop
    def run_nested(self, dlogz=None, maxiter=None, maxcall=None, add_live=True, loop='host', batch=None,
                   checkpoint_file=None, checkpoint_every=60., resume=False, on_checkpoint=None, device_init=True,
                   keep_samples=True, logl_max=None):
        """sampler.py:1214-1356 / 1040-1212 (no plateau mode: continuous likelihoods).

        loop='host'   : the reference's semantics -- one worst point per iteration, replacements
                        popped from a queue of `queue_size` proposals (sampler.py:732-778).
        loop='device' : the WHOLE run is rounds on the device (csrc/b2n_ns.cu, ``b2n_ns_run``): each round
                        removes the `batch` lowest live points at once and replaces them with `batch`
                        chains evolved at the threshold of the batch-th lowest -- prior draws until the
                        first bound is due (UnitCubeSampler, sampler.py:407-409), then the inner sampler.
                        No stale-threshold filter, hence no selection bias for correlated chains
                        (DESIGN.md 9.4), no host round trip per iteration.  batch defaults to
                        nlive // 40 (rwalk) or nlive // 10 (slices).
        on_checkpoint : callable(k) invoked after the k-th checkpoint has been written.
        logl_max      : stop once the lowest live point is above it (sampler.py:1103-1106; the end of a dynamic batch).
        keep_samples  : loop='device' only.  False = the positions of the dead points are NOT brought back from the
                        device (results.samples / samples_u are then empty; logz, logzerr, logl, logvol, logwt and the
                        call counts are complete): for ensembles that only want evidences.
        device_init   : False = the phase before the first bound runs in the host loop (queue of prior draws
                        evaluated on the GPU) and the device takes over when the first bound exists."""
        if resume:
            return self._resume(checkpoint_file, checkpoint_every)
        if loop not in ('host', 'device'):
            raise ValueError("loop must be 'host' or 'device'")
        if checkpoint_file is not None and loop != 'device':
            raise ValueError("checkpointing is implemented for loop='device'")
        if loop == 'device' and self.comm is not None:
            raise ValueError("loop='device' runs on one GPU (replicas: dynesty_b200.replicas)")
        if loop == 'device' and self.internal_sampler_next is None:
            raise ValueError("loop='device' needs one of the B200 samplers")
        nlive = self.nlive
        if dlogz is None:
            dlogz = 1e-3 * (nlive - 1.) + 0.01 if add_live else 0.01
        maxiter = maxiter if maxiter is not None else 1 << 62
        maxcall = maxcall if maxcall is not None else 1 << 62
        dlv = math.log((nlive + 1.) / nlive)
        half_term = math.log(0.5 * (math.exp(dlv) - 1.0))       # logsumexp([lv+dlv, lv], b=[.5,-.5]) - lv
        heap = [(float(l), i) for i, l in enumerate(self.live_logl)]
        heapq.heapify(heap)
        lmax = float(self.live_logl.max())
        logz, logvol, loglstar = LOWL, 0.0, LOWL
        cap = 4 * nlive
        dead_u = np.empty((cap, self.ndim))
        dead_v = np.empty((cap, self.ndim))
        dead_l = np.empty(cap)
        dead_nc = np.empty(cap, dtype=np.int64)
        ndead = 0
        ncall0 = self.ncall
        hand_over = False
        for it in range(1 << 62):
            delta_logz = _logaddexp(0.0, lmax + logvol - logz)
            if it > maxiter or self.ncall - ncall0 > maxcall:
                break
            if loop == 'device' and (self._q is None or self._qpos >= len(self._ql)) and \
                    (device_init or not self.unit_cube_sampling):
                hand_over = True                                    # (queue drained): the device takes over
                break
            if dlogz is not None and delta_logz < dlogz:
                break
            lnew, worst = heap[0]
            if logl_max is not None and lnew > logl_max:
                break                                              # sampler.py:1103-1106
            if lnew == lmax:
                break                                              # all live points equal: plateau
            logvol -= dlv
            # ---- _new_point (sampler.py:732-778)
            nc = 0
            while True:
                if self._q is None or self._qpos >= len(self._ql):
                    self._fill_queue(lnew)
                j = self._qpos
                self._qpos += 1
                l = self._ql[j]
                nc += self._qn[j]
                self.ncall += self._qn[j]
                if self._qpos >= len(self._ql):
                    self._queue_drained(lnew)
                if l > lnew:
                    break
            # ---- evidence increment (utils.py:1470-1492, logz part only; h/var post-hoc)
            logwt = _logaddexp(lnew, loglstar) + logvol + half_term
            logz = _logaddexp(logz, logwt)
            loglstar = lnew
            if ndead == cap:
                cap *= 2
                dead_u = np.resize(dead_u, (cap, self.ndim))
                dead_v = np.resize(dead_v, (cap, self.ndim))
                dead_l = np.resize(dead_l, cap)
                dead_nc = np.resize(dead_nc, cap)
            dead_u[ndead] = self.live_u[worst]
            dead_v[ndead] = self.live_v[worst]
            dead_l[ndead] = lnew
            dead_nc[ndead] = nc
            ndead += 1
            q = self._q
            self.live_u[worst] = q['u'][j]
            self.live_v[worst] = q['v'][j]
            self.live_logl[worst] = l
            heapq.heapreplace(heap, (l, worst))
            if l > lmax:
                lmax = l
            self.eff = 100. * self.it / self.ncall
            self.it += 1
        # ---- results (+ remaining live points, sampler.py:780-914)
        logl = dead_l[:ndead]
        logvols = -dlv * np.arange(1, ndead + 1)
        su, sv, nc_all = dead_u[:ndead], dead_v[:ndead], dead_nc[:ndead]
        if hand_over:
            # (kept on the object so that a checkpoint of the device phase carries the host phase's results)
            self._host_part = dict(su=su.copy(), sv=sv.copy(), logl=logl.copy(), logvols=logvols, nc_all=nc_all.copy(),
                                   logz=logz, logvol=logvol, loglstar=loglstar, dlogz=dlogz, add_live=add_live,
                                   maxiter=maxiter - ndead,
                                   maxcall=ncall0 + maxcall if maxcall < (1 << 61) else None)
            dev = self._device_rounds(logz, logvol, loglstar, dlogz, self._host_part['maxiter'],
                                      self._host_part['maxcall'], batch, checkpoint_file=checkpoint_file,
                                      checkpoint_every=checkpoint_every, on_checkpoint=on_checkpoint,
                                      keep_samples=keep_samples or checkpoint_file is not None, logl_max=logl_max)
            return self._finalize(su, sv, logl, logvols, nc_all, dev, add_live)
        return self._finalize(su, sv, logl, logvols, nc_all, None, add_live)

    def _resume(self, checkpoint_file, checkpoint_every):
        """Continue a run restored from a checkpoint of the device phase (``NestedSampler.restore``)."""
        snap, hp = getattr(self, '_dev_snap', None), getattr(self, '_host_part', None)
        if snap is None or hp is None:
            raise ValueError("nothing to resume: the pickle carries no snapshot of a device-resident run")
        dev = self._device_rounds(hp['logz'], hp['logvol'], hp['loglstar'], hp['dlogz'], hp['maxiter'], hp['maxcall'],
                                  snap['batch'], checkpoint_file=checkpoint_file, checkpoint_every=checkpoint_every,
                                  snap=snap)
        return self._finalize(hp['su'], hp['sv'], hp['logl'], hp['logvols'], hp['nc_all'], dev, hp['add_live'])

    def _finalize(self, su, sv, logl, logvols, nc_all, dev, add_live):
        """Results (+ remaining live points, sampler.py:780-914) from the host-phase and device-phase dead points."""
        nlive = self.nlive
        ndead = len(logl)
        have_pos = True
        if dev is not None:
            du, dv, dl, dlvol, dnc = dev
            logl, logvols = np.concatenate([logl, dl]), np.concatenate([logvols, dlvol])
            have_pos = len(du) == len(dl)
            su, sv = (np.concatenate([su, du]), np.concatenate([sv, dv])) if have_pos else (du, dv)
            nc_all = np.concatenate([nc_all, dnc.astype(np.int64)])
            ndead = len(logl)
        if add_live:
            order = np.argsort(self.live_logl)
            lv_live = np.log(1. - (np.arange(nlive) + 1.) / (nlive + 1.)) + (logvols[-1] if ndead else 0.0)
            logl = np.concatenate([logl, self.live_logl[order]])
            logvols = np.concatenate([logvols, lv_live])
            if have_pos:
                su = np.concatenate([su, self.live_u[order]])
                sv = np.concatenate([sv, self.live_v[order]])
            nc_all = np.concatenate([nc_all, np.ones(nlive, dtype=np.int64)])
        # number of live points when each sample died (results.samples_n, utils.py:1237-1270): nlive in the host loop,
        # N - j for the j-th removal of a device round, nlive - k for the k-th of the final live points
        nhost = ndead - (len(dev[2]) if dev is not None else 0)
        samples_n = np.full(ndead, nlive, dtype=np.int64)
        if dev is not None and len(dev[2]):
            samples_n[nhost:] = nlive - (np.arange(len(dev[2])) % max(1, getattr(self, 'batch', 1)))
        if add_live:
            samples_n = np.concatenate([samples_n, nlive - np.arange(nlive)])
        sh = np.array(self.scale_history, dtype=float).reshape(-1, 2)
        cum = np.cumsum(nc_all)
        sample_scale = (sh[np.minimum(np.searchsorted(sh[:, 0], cum + (self.nlive if len(cum) else 0)), len(sh) - 1), 1]
                        if len(sh) else np.ones(len(nc_all)))
        logwt, logzs, logzvar, h = _integrate(logl, logvols)
        self.results = Results(niter=ndead, ncall=int(self.ncall), eff=100. * ndead / max(self.ncall, 1),
                               samples_u=su, samples=sv, logl=logl, logvol=logvols, logwt=logwt, logz=logzs,
                               logzerr=np.sqrt(logzvar), information=h, ncall_per_it=nc_all,
                               samples_n=samples_n, samples_scale=sample_scale,
                               nbound=self.nbound, nbatches=self.nbatches, n_proposals=self.n_proposals,
                               bound_history=list(self.bound_history), scale_history=list(self.scale_history))
        return self.results
