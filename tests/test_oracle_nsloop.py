"""CPU tier: the oracle of the batched-replacement rounds (oracle/nsloop.py) and the host side of
``run_nested(loop='device')`` driven through the oracle-backed stand-in (tests/fake_backend.py).

Pins: (i) the quadrature of a round against the post-hoc integration of dynesty_b200.nested, and that
against stored outputs of the reference's own ``utils.compute_integrals``;
(ii) batch = 1 reproduces the reference's serial update rule (one point per iteration, ln X falls by
ln((N+1)/N)); (iii) logZ of whole runs against the analytic truth."""
import math
import os

import numpy as np
import pytest

from oracle import nsloop, likelihoods as OL, bounding as OB
from dynesty_b200 import likelihoods as DL, nested


def _bound_of(points, strict=True, enlarge=1.25):
    e = OB.bounding_ellipsoid(points)
    e.scale_to_logvol(e.logvol + math.log(enlarge))
    return dict(ctrs=e.ctr[None], ams=e.am[None], axes=e.axes[None], logvols=np.array([e.logvol]), strict=strict)


def _setup(N=60, K=12, sampler='rwalk', steps=8, seed=11, **kw):
    m = OL.gauss_test3d()
    rng = np.random.default_rng(5)
    u = 0.5 + 0.12 * (rng.random((N, 3)) - 0.5)
    v = m.prior_transform(u)
    l = np.array([float(m.loglike(x)) for x in v])
    b = nsloop.BatchNS(m, u, v, l, K, sampler, steps, seed, bound=_bound_of(u), logvol=-3.0, logz=-50.0,
                       loglstar=float(l.min()) - 1.0, **kw)
    return m, b



def _abort_at(k_stop):
    """on_checkpoint callback that kills the run after its k_stop-th checkpoint (the reference's
    tests/test_resume.py kills the process instead)."""
    def cb(k):
        if k >= k_stop:
            raise KeyboardInterrupt('test: run aborted after checkpoint %d' % k)
    return cb


@pytest.mark.parametrize('sampler,steps', [('rwalk', 8), ('rslice', 3), ('slice', 1), ('unif', 1)])
def test_round_invariants(sampler, steps):
    m, b = _setup(sampler=sampler, steps=steps)
    l0 = np.sort(b.live_logl)
    assert b.step()
    du, dv, dl, dlv, dnc = b.dead_arrays()
    assert len(dl) == 12 and np.all(np.diff(dl) >= 0)
    assert np.allclose(dl, l0[:12])                                  # the 12 lowest died, ascending
    # survivors untouched, replacements strictly above the threshold
    assert b.last['thr'] == l0[11] and np.all(b.live_logl > l0[11])
    assert np.isin(l0[12:], b.live_logl).all()
    # ln X after the round: ln X0 + ln((N-K+1)/(N+1))
    assert b.logvol == pytest.approx(-3.0 + math.log((60 - 12 + 1) / 61.0))
    assert np.allclose(dlv, -3.0 + np.log((60 - np.arange(12)) / 61.0))
    assert b.ncall == dnc.sum() and b.it == 12 and b.round == 1
    for x, vv, ll in zip(b.live_u, b.live_v, b.live_logl):           # (u, v, logl) stay consistent
        assert np.allclose(m.prior_transform(x), vv) and float(m.loglike(vv)) == pytest.approx(ll)


def test_quadrature_matches_posthoc_and_reference():
    """The running logZ of the rounds == the post-hoc trapezoid integral over (logl, logvol) of the dead
    points (dynesty_b200.nested._integrate) == the reference's utils.compute_integrals (its output on the dead
    points of a device-loop run, stored with them in tests/golden/dynamic.npz by oracle/make_golden.py)."""
    m, b = _setup(N=80, K=10, steps=6)
    b.logvol, b.logz, b.loglstar = 0.0, -1e300, -1e300
    for _ in range(6):
        assert b.step()
        b.bound = _bound_of(b.live_u)
    _, _, dl, dlv, _ = b.dead_arrays()
    logwt, logz, _, _ = nested._integrate(dl, dlv)
    assert logz[-1] == pytest.approx(b.logz, rel=1e-12)
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'dynamic.npz'))
    logwt, logz, _, _ = nested._integrate(g['logl'], g['logvol'])
    np.testing.assert_allclose(logz, g['integrals_logz'], rtol=1e-12)     # (saved_logwt, saved_logz, var, h)
    np.testing.assert_allclose(logwt, g['integrals_logwt'], rtol=1e-12)


def test_batch_one_is_the_serial_rule():
    m, b = _setup(N=40, K=1, steps=5)
    lv0 = b.logvol
    worst = float(b.live_logl.min())
    assert b.step()
    assert b.dead['logl'] == [worst]
    assert b.logvol == pytest.approx(lv0 - math.log(41 / 40.))        # sampler.py:1131: dlv = ln((N+1)/N)
    assert b.loglstar == worst and b.live_logl.min() > worst


def test_stop_flags():
    m, b = _setup(update_interval=50)
    assert b.step() and b.need_bound == 1 and not b.step()            # 12 chains x 8 walks = 96 >= 50
    b.bound_updated(_bound_of(b.live_u))
    assert b.need_bound == 0 and b.ncall_last_update == b.ncall and b.step()
    b.bound_updated(_bound_of(b.live_u))
    tight = dict(b.bound)                                             # a bound that excludes every live point
    tight['ctrs'] = b.bound['ctrs'] + 10.0
    b.bound = tight
    assert not b.step() and b.need_bound == 2
    m, b = _setup(dlogz=1e9)
    assert not b.step() and b.done == 1


@pytest.mark.parametrize('sample,kw', [('rwalk', dict(walks=12)), ('rslice', dict(slices=3)), ('unif', dict(bootstrap=0))])
def test_device_loop_host_logic_logz(fake_ops, sample, kw):
    """run_nested(loop='device') end to end on the oracle backend: prior-draw rounds until the first bound is
    due, rounds + bound updates (fitted where the live points lie: ns_update_bound), results integration; logZ
    against the analytic truth."""
    m = DL.gauss_test3d()
    s = nested.NestedSampler(m, nlive=120, bound='multi', sample=sample, queue_size=40, seed=3, **kw)
    res = s.run_nested(dlogz=0.5, loop='device', batch=24)
    truth = 3 * (-np.log(20.))
    assert abs(res.logz[-1] - truth) < 4 * res.logzerr[-1] + 0.05
    assert s.device_rounds > 10 and s.nbound > 2 and not s.unit_cube_sampling
    assert np.all(np.diff(res.logl) >= 0)                             # dead points ascending
    assert np.all(np.diff(res.logvol) < 0)
    assert res.ncall == s.ncall and res.ncall_per_it.sum() <= res.ncall
    mean, cov = res.posterior_moments()
    assert np.all(np.abs(mean - np.linspace(-1, 1, 3)) < 0.4)


def test_device_loop_without_bound_and_rejections(fake_ops):
    """bound='none' (the reference then samples the unit cube for the whole run, sampler.py:625-674): the device
    rounds stay in the prior-draw phase; a multi-rank communicator is refused (replicas shard, rounds do not)."""
    m = DL.gauss_test3d()
    s = nested.NestedSampler(m, nlive=50, bound='none', sample='unif', seed=4)
    res = s.run_nested(loop='device', batch=5, dlogz=None, maxiter=60)
    assert s.unit_cube_sampling and s.nbound == 1 and 60 <= res.niter < 60 + 5
    assert np.all(np.diff(res.logl[:res.niter]) >= 0)
    s2 = nested.NestedSampler(m, nlive=50, bound='multi', sample='rwalk', seed=4)
    s2.comm = object()
    with pytest.raises(ValueError):
        s2.run_nested(loop='device')


@pytest.mark.parametrize('sample,kw', [('rwalk', dict(walks=12)), ('rslice', dict(slices=3))])
def test_checkpoint_resume_is_bit_identical(fake_ops, tmp_path, sample, kw):
    """The reference's tests/test_resume.py property: a run killed after a checkpoint and resumed from the file
    ends with the SAME results as the uninterrupted run (utils.py:2321-2355 save / restore).  Here the checkpoint
    carries the snapshot of the device-resident phase (live set, scalars, round counter, dead rows so far)."""
    m = DL.gauss_test3d()
    mk = lambda: nested.NestedSampler(m, nlive=100, bound='multi', sample=sample, queue_size=25, seed=11, **kw)
    ref = mk().run_nested(dlogz=0.5, loop='device', batch=20)
    f = str(tmp_path / 'ckpt.pkl')
    s = mk()
    with pytest.raises(KeyboardInterrupt):
        s.run_nested(dlogz=0.5, loop='device', batch=20, checkpoint_file=f, checkpoint_every=0., on_checkpoint=_abort_at(3))
    del s
    r = nested.NestedSampler.restore(f)
    assert r._dev_snap is not None and r._dev_snap['rounds'] > 0 and len(r._dev_snap['dead'][2]) > 0
    res = r.run_nested(resume=True)
    assert res.niter == ref.niter and res.ncall == ref.ncall and r.nbound == 1 + len(ref.bound_history)
    assert np.array_equal(res.logl, ref.logl) and np.array_equal(res.logvol, ref.logvol)
    assert np.array_equal(res.samples_u, ref.samples_u)
    assert res.logz[-1] == ref.logz[-1]
    with pytest.raises(ValueError):
        mk().run_nested(resume=True)


def test_device_loop_single_bound_and_limits(fake_ops):
    """bound='single' (non-strict contains) inside the rounds; maxiter / maxcall stop the device phase."""
    m = DL.gauss_test3d()
    s = nested.NestedSampler(m, nlive=100, bound='single', sample='rwalk', walks=10, queue_size=25, seed=5)
    res = s.run_nested(dlogz=0.5, loop='device', batch=10)
    assert abs(res.logz[-1] - 3 * (-np.log(20.))) < 4 * res.logzerr[-1] + 0.1
    assert s.device_rounds > 5 and isinstance(s.bound, type(s.bound_next))
    s2 = nested.NestedSampler(m, nlive=100, bound='single', sample='rwalk', walks=10, queue_size=25, seed=5)
    r2 = s2.run_nested(dlogz=None, maxiter=400, loop='device', batch=10, add_live=False)
    assert 400 <= r2.niter <= 400 + 10                  # checked once per round
    s3 = nested.NestedSampler(m, nlive=100, bound='single', sample='rwalk', walks=10, queue_size=25, seed=5)
    r3 = s3.run_nested(dlogz=None, maxcall=6000, loop='device', batch=10, add_live=False)
    assert r3.ncall <= 100 + 6000 + 10 * 10 + 25 * 10


def test_replicas_plumbing(fake_ops):
    """dynesty_b200.replicas: one device-resident run per seed; a replica equals the same run done on its own
    (the oracle backend has ONE device state, so the replicas run one at a time here; on the GPU every replica
    owns a context and they run concurrently -- tests/test_gpu_replicas.py)."""
    from dynesty_b200 import replicas
    m = DL.gauss_test3d()
    kw = dict(nlive=80, bound='multi', sample='rwalk', sampler_kwargs=dict(walks=10), max_in_flight=1, dlogz=0.5, batch=16)
    outs, wall = replicas.run_replicas(m, [3, 4, 5], **kw)
    assert [o['seed'] for o in outs] == [3, 4, 5] and wall > 0
    s = nested.NestedSampler(m, nlive=80, bound='multi', sample='rwalk', walks=10, seed=4)
    r = s.run_nested(loop='device', dlogz=0.5, batch=16)
    assert outs[1]['logz'] == float(r.logz[-1]) and outs[1]['ncall'] == r.ncall
    summ = replicas.summarize(outs, wall)
    assert summ['replicas'] == 3 and summ['ncall'] == sum(o['ncall'] for o in outs)
    assert abs(summ['logz_mean'] - 3 * (-np.log(20.))) < 1.0
