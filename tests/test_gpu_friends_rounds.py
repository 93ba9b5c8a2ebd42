"""GPU tier: RadFriends / SupFriends bounds inside the device-resident rounds (friends mode of csrc/b2n_ns.cu:
b2n_ns_update_friends / _set_friends / _get_friends, device-paced friends_unif_kernel).

Tolerances (as tests/test_gpu_nsloop.py): dead-point order, per-chain ncall and call totals exact; ln X 1e-13;
running logZ 1e-10; live set rtol 1e-8.  The device update against the host route: bit-identical."""
import math

import numpy as np
import pytest

from oracle import likelihoods as OL, friends as OF
from friends_rounds_oracle import FriendsBatchNS, FRIENDS_BOOT_CHAIN, friends_boot_idxs
from dynesty_b200 import ops, likelihoods as DL, nested, bounding as B

pytestmark = pytest.mark.gpu
SEED = 56432


def _models(kind, n):
    if kind == 'gauss':
        return DL.gauss_corr(n, 0.4, 5.0), OL.gauss_corr(n, 0.4, 5.0)
    return DL.shells(n), OL.shells(n)


def _live(om, n, N, rng, two=False):
    if two:                 # two separated blobs around the two shell centres (several clusters under the cubes' metric)
        half = N // 2
        c1, c2 = 0.5 + np.zeros(n), 0.5 + np.zeros(n)
        c1[0], c2[0] = 0.5 - 3.5 / 12, 0.5 + 3.5 / 12
        u = np.concatenate([c1 + 0.03 * rng.standard_normal((half, n)), c2 + 0.03 * rng.standard_normal((N - half, n))])
    else:
        u = 0.5 + 0.05 * rng.standard_normal((N, n))
    v = om.prior_transform(u)
    l = np.array([float(om.loglike(x)) for x in v])
    return u, v, l


def _compare(st, o, N, n, K, rounds):
    assert (st['done'], st['need_bound'], st['error']) == (0, 0, 0), st
    assert st['rounds'] == o.round and st['it'] == o.it and st['ncall'] == o.ncall
    du, dv, dl, dlv, dnc = ops.ns_get_dead(0, st['it'], n)
    ou, ov, ol, olv, onc = o.dead_arrays()
    assert np.array_equal(dl[:K], ol[:K])
    assert np.allclose(dl, ol, rtol=1e-9, atol=0) and np.allclose(du, ou, rtol=1e-8, atol=1e-12)
    assert np.allclose(dlv, olv, rtol=0, atol=1e-13)
    assert np.array_equal(dnc, onc)
    lu, lv_, ll = ops.ns_get_live(N, n)
    pd, po = np.argsort(ll, kind='stable'), np.argsort(o.live_logl, kind='stable')
    assert np.allclose(ll[pd], o.live_logl[po], rtol=1e-8, atol=1e-10)
    assert np.allclose(lu[pd], o.live_u[po], rtol=1e-8, atol=1e-12)
    assert st['logz'] == pytest.approx(o.logz, rel=1e-10)
    assert st['logvol'] == pytest.approx(o.logvol, abs=1e-13)
    assert st['scale'] == pytest.approx(o.scale, rel=1e-10)


def _start(dm, om, fkind, n, N, K, sampler, steps, rounds, two=False, flags=None, seed_live=0):
    rng = np.random.default_rng(300 + n + K + seed_live)
    u, v, l = _live(om, n, N, rng, two)
    f = OF.Friends(n, fkind)
    f.update(u)
    chain0, scale0 = 1000, 0.7
    o = FriendsBatchNS(om, u, v, l, K, sampler, steps, SEED, chain0=chain0, scale=scale0, logvol=-2.5, logz=-40.0,
                       loglstar=float(l.min()) - 0.5, ncall=500, friends=f, dlogz=1e-9, dimflags=flags)
    ops.ns_create(dm.model_id(), N, n, K, ('rwalk', 'rslice', 'slice', 'unif').index(sampler), steps, SEED,
                  chain0=chain0, dlogz=1e-9, dead_capacity=4 * rounds * K + 5,
                  dimflags=None if flags is None else np.array(flags, dtype=np.uint8))
    ops.ns_set_state(u, v, l, -2.5, -40.0, float(l.min()) - 0.5, 500, scale0)
    ops.ns_set_friends(fkind, f.cov, f.am, f.axes, f.axes_inv, f.logvol)
    return o, f


CASES = [
    # model, bound kind, n, N, K, sampler, steps, rounds, dimflags
    ('gauss', 'balls', 2, 60, 1, 'unif', 1, 12, None),
    ('gauss', 'cubes', 3, 120, 8, 'unif', 1, 4, None),
    ('shells', 'balls', 5, 200, 8, 'unif', 1, 3, None),
    ('gauss', 'balls', 3, 100, 8, 'rwalk', 10, 3, None),
    ('gauss', 'cubes', 5, 150, 1, 'rwalk', 10, 8, None),
    ('gauss', 'balls', 2, 80, 8, 'rslice', 3, 3, None),
    ('gauss', 'cubes', 5, 200, 8, 'rslice', 4, 3, None),
    ('gauss', 'balls', 3, 100, 8, 'rwalk', 10, 3, [1, 2, 0]),      # periodic / reflective dims
    ('gauss', 'cubes', 3, 100, 8, 'unif', 1, 3, [1, 2, 0]),
]


@pytest.mark.parametrize('kind,fkind,n,N,K,sampler,steps,rounds,flags', CASES)
def test_friends_rounds_match_oracle(kind, fkind, n, N, K, sampler, steps, rounds, flags):
    dm, om = _models(kind, n)
    o, f = _start(dm, om, fkind, n, N, K, sampler, steps, rounds, flags=flags)
    try:
        for _ in range(rounds):
            assert o.step(), (o.done, o.need_bound)
        st = ops.ns_run(rounds, 0)
        _compare(st, o, N, n, K, rounds)
    finally:
        ops.ns_destroy()


@pytest.mark.parametrize('kind,fkind,n,N,K,sampler,steps,nboot,enlarge,two', [
    ('shells', 'cubes', 3, 120, 8, 'unif', 1, 0, 1.0, True),        # two blobs: nclusters > 1, leave-one-out radius
    ('shells', 'cubes', 3, 120, 8, 'unif', 1, 5, 1.0, True),        # ... bootstrap radius
    ('gauss', 'balls', 2, 80, 8, 'unif', 1, 3, 1.0, False),
    ('gauss', 'balls', 3, 100, 8, 'rwalk', 10, 0, 1.25, False),
    ('gauss', 'cubes', 2, 80, 4, 'rslice', 3, 3, 1.0, False),
])
def test_friends_rounds_straddling_a_device_update(kind, fkind, n, N, K, sampler, steps, nboot, enlarge, two):
    dm, om = _models(kind, n)
    o, f = _start(dm, om, fkind, n, N, K, sampler, steps, 6, two=two)
    try:
        for _ in range(3):
            assert o.step()
        st = ops.ns_run(3, 0)
        _compare(st, o, N, n, K, 3)
        # the oracle's update at the same round, with the documented bootstrap streams
        g = OF.Friends(n, fkind)
        g.am = f.am.copy()
        ncl = int(OF.components_within(o.live_u, g.am).max()) + 1
        r = g.update(o.live_u, bootstrap_idxs=friends_boot_idxs(SEED, o.round, nboot, N))
        if enlarge != 1.0:
            g.scale_to_logvol(g.logvol + math.log(enlarge))
        lv, rad, dncl = ops.ns_update_friends(fkind, enlarge, nboot)
        assert dncl == ncl and rad == pytest.approx(r, rel=1e-8) and lv == pytest.approx(g.logvol, rel=1e-9, abs=1e-9)
        if two:
            assert dncl > 1
        ops.ns_bound_updated()
        o.bound_updated(g)
        for _ in range(3):
            assert o.step()
        st = ops.ns_run(3, 0)
        _compare(st, o, N, n, K, 6)
    finally:
        ops.ns_destroy()


@pytest.mark.parametrize('fkind,nboot,enlarge,two', [('cubes', 0, 1.0, True), ('cubes', 4, 1.0, True),
                                                     ('balls', 0, 1.3, False), ('balls', 2, 1.0, False)])
def test_device_update_equals_host_route(fkind, nboot, enlarge, two):
    """ns_update_friends == ops.friends_update on the run's live set (same am_prev, nboot, seed, chain ids) followed by
    the host class's scale_to_logvol: every output bit-identical."""
    n, N, K = 3, 120, 8
    dm, om = _models('shells', n)
    o, f = _start(dm, om, fkind, n, N, K, 'unif', 1, 2, two=two)
    try:
        st = ops.ns_run(2, 0)
        assert st['rounds'] == 2
        prev = ops.ns_get_friends(n)
        assert np.array_equal(prev['am'], f.am) and math.isnan(prev['radius']) and prev['nclusters'] == 0
        live = ops.ns_get_live(N, n, only_u=True)
        h = ops.friends_update(live, fkind, am_prev=prev['am'], use_clustering=True, nboot=nboot, seed=SEED,
                               chain0=FRIENDS_BOOT_CHAIN + (st['rounds'] << 8))
        hb = (B.B200RadFriends if fkind == 'balls' else B.B200SupFriends)(n)
        hb.cov, hb.am, hb.axes, hb.axes_inv, hb.logvol = h['cov'], h['am'], h['axes'], h['axes_inv'], h['logvol']
        if enlarge != 1.0:
            hb.scale_to_logvol(hb.logvol + math.log(enlarge))
        lv, rad, ncl = ops.ns_update_friends(fkind, enlarge, nboot)
        d = ops.ns_get_friends(n)
        for k in ('cov', 'am', 'axes', 'axes_inv'):
            assert np.array_equal(d[k], getattr(hb, k)), k
        assert d['logvol'] == hb.logvol == lv
        assert d['radius'] == h['radius'] == rad and d['nclusters'] == h['nclusters'] == ncl
        if two:
            assert ncl > 1
    finally:
        ops.ns_destroy()


def test_nboot_above_255_is_refused():
    dm, om = _models('gauss', 2)
    o, f = _start(dm, om, 'balls', 2, 40, 4, 'unif', 1, 1)
    try:
        with pytest.raises(ValueError):
            ops.ns_update_friends('balls', 1.0, 256)
    finally:
        ops.ns_destroy()


def _check_run(s, res, truth):
    assert abs(res.logz[-1] - truth) < 4 * res.logzerr[-1] + 0.1, (res.logz[-1], res.logzerr[-1], truth)
    assert s.device_rounds > 10 and s.nbound > 2 and not s.unit_cube_sampling
    assert s.bound.ctrs is s.live_u
    assert s.bound.contains_many(s.live_u).all()
    assert all(h[1] == 1 for h in s.bound_history)


@pytest.mark.parametrize('bound,sample,kw', [('balls', 'unif', {}), ('cubes', 'unif', {}),
                                              ('balls', 'rwalk', dict(walks=15)), ('cubes', 'rwalk', dict(walks=15))])
def test_device_loop_gauss3d(bound, sample, kw):
    m = DL.gauss_test3d()
    s = nested.NestedSampler(m, nlive=300, bound=bound, sample=sample, seed=7, **kw)
    res = s.run_nested(dlogz=0.5, loop='device')
    _check_run(s, res, m.logz_truth)


@pytest.mark.parametrize('name,bound', [('shells', 'balls'), ('shells', 'cubes'), ('eggbox', 'balls')])
def test_device_loop_multimodal_2d(name, bound):
    m = DL.shells(2) if name == 'shells' else DL.eggbox(2)
    s = nested.NestedSampler(m, nlive=500, bound=bound, sample='unif', seed=11)
    res = s.run_nested(dlogz=0.2, loop='device')
    _check_run(s, res, m.logz_truth)


def _abort_at(k_stop):
    def cb(k):
        if k >= k_stop:
            raise KeyboardInterrupt('test: run aborted after checkpoint %d' % k)
    return cb


@pytest.mark.parametrize('bound,sample,kw', [('balls', 'unif', {}), ('cubes', 'rwalk', dict(walks=12, enlarge=1.25))])
def test_checkpoint_resume_is_bit_identical(tmp_path, bound, sample, kw):
    m = DL.gauss_test3d()
    mk = lambda: nested.NestedSampler(m, nlive=200, bound=bound, sample=sample, seed=13, **kw)
    ref = mk().run_nested(dlogz=0.5, loop='device', batch=10)
    f = str(tmp_path / 'ckpt.pkl')
    s = mk()
    with pytest.raises(KeyboardInterrupt):
        s.run_nested(dlogz=0.5, loop='device', batch=10, checkpoint_file=f, checkpoint_every=0., on_checkpoint=_abort_at(2))
    del s
    r = nested.NestedSampler.restore(f)
    assert r._dev_snap is not None and r._dev_snap['rounds'] > 0
    res = r.run_nested(resume=True)
    assert res.niter == ref.niter and res.ncall == ref.ncall
    assert np.array_equal(res.logl, ref.logl) and np.array_equal(res.samples_u, ref.samples_u)
    assert res.logz[-1] == ref.logz[-1]


def test_replicas_and_dynamic_with_balls():
    from dynesty_b200 import replicas, dynamic as D
    m = DL.gauss_test3d()
    kw = dict(nlive=200, bound='balls', sample='unif', dlogz=0.5)
    outs, _ = replicas.run_replicas(m, [21, 22, 23], max_in_flight=3, **kw)
    solo, _ = replicas.run_replicas(m, [22], max_in_flight=1, **kw)
    assert (outs[1]['logz'], outs[1]['ncall'], outs[1]['niter'], outs[1]['nbound']) == \
        (solo[0]['logz'], solo[0]['ncall'], solo[0]['niter'], solo[0]['nbound'])
    assert len({o['logz'] for o in outs}) == 3
    d = D.DynamicNestedSampler(m, nlive=200, bound='balls', sample='unif', seed=5)
    res = d.run_nested(maxbatch=2, n_effective=1e9)
    assert d.batch == 2 and np.all(np.diff(res.logl) >= 0)
    assert abs(res.logz[-1] - m.logz_truth) < 4 * res.logzerr[-1] + 0.1
