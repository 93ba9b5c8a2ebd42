"""CPU tier: RadFriends / SupFriends bounds inside the device-resident rounds.

(i) The oracle of the rounds with an ``oracle.friends.Friends`` bound (tests/friends_rounds_oracle.py, on top of
oracle/nsloop.py): round invariants, batch = 1 is the serial rule, the forced update (need_bound = 2) never fires.
(ii) The host side of ``run_nested(loop='device')`` with bound='balls' / 'cubes' on the oracle backend (tests/fake_backend.py), with stand-ins for the three friends entry
points of the rounds (b2n_ns_update_friends / _set_friends / _get_friends) defined here on top of it."""
import math

import numpy as np
import pytest

from oracle import likelihoods as OL, friends as OF
from friends_rounds_oracle import FriendsBatchNS, friends_boot_idxs
from dynesty_b200 import likelihoods as DL, nested, bounding as B

TRUTH3 = 3 * (-np.log(20.))


def _friends_of(points, kind='balls', enlarge=1.0):
    f = OF.Friends(points.shape[1], kind)
    f.update(points)
    if enlarge != 1.0:
        f.scale_to_logvol(f.logvol + math.log(enlarge))
    return f


def _setup(N=60, K=12, sampler='rwalk', steps=8, seed=11, kind='balls', **kw):
    m = OL.gauss_test3d()
    rng = np.random.default_rng(5)
    u = 0.5 + 0.12 * (rng.random((N, 3)) - 0.5)
    v = m.prior_transform(u)
    l = np.array([float(m.loglike(x)) for x in v])
    b = FriendsBatchNS(m, u, v, l, K, sampler, steps, seed, friends=_friends_of(u, kind), logvol=-3.0, logz=-50.0,
                       loglstar=float(l.min()) - 1.0, **kw)
    return m, b


@pytest.mark.parametrize('kind', ['balls', 'cubes'])
@pytest.mark.parametrize('sampler,steps', [('rwalk', 8), ('rslice', 3), ('unif', 1)])
def test_friends_round_invariants(kind, sampler, steps):
    m, b = _setup(sampler=sampler, steps=steps, kind=kind)
    l0 = np.sort(b.live_logl)
    live0 = b.live_u.copy()
    assert b.step()
    du, dv, dl, dlv, dnc = b.dead_arrays()
    assert len(dl) == 12 and np.allclose(dl, l0[:12])
    assert b.last['thr'] == l0[11] and np.all(b.live_logl > l0[11])
    assert np.isin(l0[12:], b.live_logl).all()
    assert b.ncall == dnc.sum() and b.it == 12 and b.round == 1 and b.need_bound == 0
    if sampler == 'unif':                     # centres of the round = the live set at its start (worst points included)
        assert np.array_equal(b.friends.ctrs, live0)
    for x, vv, ll in zip(b.live_u, b.live_v, b.live_logl):
        assert np.allclose(m.prior_transform(x), vv) and float(m.loglike(vv)) == pytest.approx(ll)


def test_friends_batch_one_is_the_serial_rule():
    m, b = _setup(N=40, K=1, sampler='unif', steps=1)
    lv0, worst = b.logvol, float(b.live_logl.min())
    assert b.step()
    assert b.dead['logl'] == [worst]
    assert b.logvol == pytest.approx(lv0 - math.log(41 / 40.))
    assert b.loglstar == worst and b.live_logl.min() > worst


def test_friends_never_force_an_update():
    """A start point is a centre of the bound: even a bound whose shape excludes every other point (a tiny radius)
    contains it, so sampler.py:485-489 cannot fire -- need_bound is never 2."""
    m, b = _setup(sampler='rwalk', steps=4)
    f = b.friends
    f.scale_to_logvol(f.logvol - 30.0)
    b.use(f)
    f.ctrs = b.live_u
    for _ in range(4):
        assert all(f.contains(b.live_u[i]) for i in range(b.N))
        assert b.step()
        assert b.need_bound != 2


def test_friends_boot_chain_ids():
    idx = friends_boot_idxs(7, 3, 2, 50)
    assert len(idx) == 2 and all(len(i) == 50 and i.min() >= 0 and i.max() < 50 for i in idx)
    from oracle import philox
    assert np.array_equal(idx[1], philox.ChainStream(7, 0x6000000000000000 + (3 << 8) + 1).integers(50, 50))
    assert friends_boot_idxs(7, 3, 0, 50) is None


# ---- the three friends entry points of the rounds on the oracle backend ------------------------------------------
@pytest.fixture
def fake_friends(fake_ops, monkeypatch):
    from dynesty_b200 import ops
    st = fake_ops._state
    create0 = fake_ops.ns_create

    def ns_create(*a, **k):
        st.pop('ns_friends', None)
        return create0(*a, **k)

    def ns_set_state(live_u, live_v, live_logl, logvol, logz, loglstar, ncall, scale, ctx=None):
        c = st['ns_cfg']        # (fake_backend.ns_set_state, with the friends-aware rounds)
        st['ns'] = FriendsBatchNS(c['model'], live_u, live_v, live_logl, c['batch'], c['sampler'], c['steps'],
                                  c['seed'], chain0=c['chain0'], facc=c['facc'], scale=scale, logvol=logvol,
                                  logz=logz, loglstar=loglstar, ncall=ncall, update_interval=c['update_interval'],
                                  dlogz=c['dlogz'], maxiter=c['maxiter'], maxcall=c['maxcall'], bound=None,
                                  unit_cube_phase=c['unit_cube_phase'], first_min_ncall=c['first_min_ncall'],
                                  first_min_eff=c['first_min_eff'], it0=c['it0'], logl_max=c['logl_max'])

    def _bound():
        return st['ns_friends'][0] if 'ns_friends' in st else fake_ops._ns_bound()

    def ns_run(max_rounds, check_every=0, ctx=None):
        b = st['ns']
        if b.phase == 1:
            if 'ns_friends' in st:
                b.use(st['ns_friends'][0])
            else:
                b.bound = fake_ops._ns_bound()
        for _ in range(max_rounds):
            if not b.step():
                break
        return fake_ops.ns_status()

    def ns_bound_updated(ctx=None):
        st['ns'].bound_updated(_bound())

    def ns_update_friends(kind, enlarge=1.0, nboot=0, use_clustering=True, ctx=None):
        b = st['ns']
        if nboot > 255:
            raise ValueError('nboot <= 255')
        f = OF.Friends(b.n, kind)
        if 'ns_friends' in st:                                     # am_prev: the run's current metric
            f.am = st['ns_friends'][0].am.copy()
        ncl = int(OF.components_within(b.live_u, f.am).max()) + 1 if use_clustering else 1
        r = f.update(b.live_u, bootstrap_idxs=friends_boot_idxs(b.seed, b.round, nboot, b.N),
                     use_clustering=use_clustering)
        if enlarge != 1.0:
            f.scale_to_logvol(f.logvol + math.log(enlarge))
        st['ns_friends'] = (f, r, ncl)
        st['ns_friends_calls'] = st.get('ns_friends_calls', 0) + 1
        return float(f.logvol), r, ncl

    def ns_set_friends(kind, cov, am, axes, axes_inv, logvol, ctx=None):
        b = st['ns']
        f = OF.Friends(b.n, kind)
        f.cov, f.am, f.axes, f.axes_inv = (np.array(a, dtype=float) for a in (cov, am, axes, axes_inv))
        f.logvol, f.ctrs = float(logvol), b.live_u
        st['ns_friends'] = (f, math.nan, 0)

    def ns_get_friends(ndim, ctx=None):
        f, r, ncl = st['ns_friends']
        return dict(cov=f.cov.copy(), am=f.am.copy(), axes=f.axes.copy(), axes_inv=f.axes_inv.copy(),
                    logvol=float(f.logvol), radius=r, nclusters=ncl)

    for name, fn in dict(ns_create=ns_create, ns_set_state=ns_set_state, ns_run=ns_run, ns_bound_updated=ns_bound_updated,
                         ns_update_friends=ns_update_friends, ns_set_friends=ns_set_friends,
                         ns_get_friends=ns_get_friends).items():
        monkeypatch.setattr(ops, name, fn)
    return fake_ops


@pytest.mark.parametrize('bound,sample,kw', [('balls', 'unif', {}), ('cubes', 'unif', dict(bootstrap=0)),
                                              ('balls', 'rwalk', dict(walks=10)), ('cubes', 'rwalk', dict(walks=10))])
def test_friends_device_loop_logz(fake_friends, bound, sample, kw):
    m = DL.gauss_test3d()
    s = nested.NestedSampler(m, nlive=100, bound=bound, sample=sample, queue_size=25, seed=3, **kw)
    res = s.run_nested(dlogz=0.5, loop='device', batch=10)
    assert abs(res.logz[-1] - TRUTH3) < 4 * res.logzerr[-1] + 0.1
    assert s.device_rounds > 10 and s.nbound > 2 and not s.unit_cube_sampling
    assert isinstance(s.bound, (B.B200RadFriends, B.B200SupFriends)) and s.bound.kind == bound
    assert s.bound.ctrs is s.live_u
    assert all(h[1] == 1 for h in s.bound_history)
    assert fake_friends._state['ns_friends_calls'] == len(s.bound_history)
    f = fake_friends._state['ns_friends'][0]                        # the host object IS the device bound
    assert np.array_equal(s.bound.am, f.am) and s.bound.logvol == f.logvol
    assert s.bound.version != fake_friends._fake_ctx.resident_key and \
        s.bound.version != fake_friends._fake_ctx.friends_key


def _abort_at(k_stop):
    def cb(k):
        if k >= k_stop:
            raise KeyboardInterrupt('test: run aborted after checkpoint %d' % k)
    return cb


@pytest.mark.parametrize('bound,sample,kw', [('balls', 'unif', {}), ('cubes', 'rwalk', dict(walks=10, enlarge=1.25))])
def test_friends_checkpoint_resume_is_bit_identical(fake_friends, tmp_path, bound, sample, kw):
    m = DL.gauss_test3d()
    mk = lambda: nested.NestedSampler(m, nlive=80, bound=bound, sample=sample, queue_size=20, seed=11, **kw)
    ref_s = mk()
    ref = ref_s.run_nested(dlogz=0.5, loop='device', batch=10)
    f = str(tmp_path / 'ckpt.pkl')
    s = mk()
    with pytest.raises(KeyboardInterrupt):
        s.run_nested(dlogz=0.5, loop='device', batch=10, checkpoint_file=f, checkpoint_every=0., on_checkpoint=_abort_at(2))
    del s
    r = nested.NestedSampler.restore(f)
    assert r._dev_snap is not None and r._dev_snap['rounds'] > 0
    assert np.array_equal(r.bound.ctrs, r._dev_snap['live'][0])     # the pickled bound is the device's, centred there
    res = r.run_nested(resume=True)
    assert res.niter == ref.niter and res.ncall == ref.ncall
    assert np.array_equal(res.logl, ref.logl) and np.array_equal(res.samples_u, ref.samples_u)
    assert res.logz[-1] == ref.logz[-1]
    assert np.array_equal(r.bound.am, ref_s.bound.am) and r.bound.logvol == ref_s.bound.logvol


def test_friends_device_loop_refusals(fake_friends):
    m = DL.gauss_test3d()
    s = nested.NestedSampler(m, nlive=60, bound='balls', sample='unif', bootstrap=256, seed=2)
    with pytest.raises(ValueError):
        s.run_nested(loop='device', batch=6)
    with pytest.raises(ValueError):
        nested.NestedSampler(m, nlive=60, bound='balls', sample='rwalk', ncdim=2, seed=2)
    s2 = nested.NestedSampler(m, nlive=60, bound='cubes', sample='rwalk', seed=2)
    s2.comm = object()
    with pytest.raises(ValueError):
        s2.run_nested(loop='device')
