"""CPU tier: the B200 bounds / samplers / pool plugged into the UNMODIFIED reference
``dynesty.NestedSampler`` through its official seams (bound= / sample= / pool=), the same
way the reference's tests/test_bound_interface.py and tests/test_sampler_interface.py
plug in user classes.  Numerics come from the oracle-backed stand-in (tests/fake_backend.py);
what is pinned is the interface contract.  The tests that run the reference skip where neither a dynesty
checkout nor its copy oracle/_ref is present (oracle/refshim.py).
"""
import numpy as np
import pytest

from oracle import refshim

@pytest.fixture(scope='module')
def dynesty():
    if not refshim.available():
        pytest.skip("reference not present")
    return refshim.import_reference()


def _classes():
    # import AFTER the reference so that the mirrors subclass dynesty's own base classes
    import importlib
    import dynesty_b200._compat as c
    importlib.reload(c)
    import dynesty_b200.bounding as b
    import dynesty_b200.samplers as s
    importlib.reload(b)
    importlib.reload(s)
    return c, b, s


@pytest.mark.parametrize('bound,sample', [('multi', 'rwalk'), ('single', 'rslice'), ('multi', 'slice'),
                                          ('multi', 'unif')])
def test_dropin_run(dynesty, fake_ops, bound, sample):
    c, b, s = _classes()
    assert c.HAVE_DYNESTY
    from dynesty_b200 import likelihoods as DL
    from dynesty_b200.pool import B200Pool
    from dynesty import bounding as RB, internal_samplers as RIS
    m = DL.gauss_test3d()
    bnd = {'multi': b.B200MultiEllipsoid, 'single': b.B200Ellipsoid}[bound](3)
    smp = {'rwalk': lambda: s.B200RWalkSampler(model=m, walks=10),
           'rslice': lambda: s.B200RSliceSampler(model=m, slices=3),
           'slice': lambda: s.B200SliceSampler(model=m, slices=2),
           'unif': lambda: s.B200UniformSampler(model=m)}[sample]()
    assert isinstance(bnd, RB.Bound) and isinstance(smp, RIS.InternalSampler)
    rstate = np.random.default_rng(56432)
    ns = dynesty.NestedSampler(m.loglikelihood, m.prior_transform, 3, nlive=100, bound=bnd, sample=smp,
                               pool=B200Pool(32), queue_size=32, rstate=rstate, bootstrap=0,
                               use_pool={'prior_transform': False, 'loglikelihood': False})
    ns.run_nested(dlogz=0.5, print_progress=False)
    res = ns.results
    truth = 3 * (-np.log(20.))
    assert abs(res['logz'][-1] - truth) < 5 * res['logzerr'][-1] + 0.1
    assert ns.nbound > 1                                   # the B200 bound was updated by Sampler
    assert isinstance(ns.bound, type(bnd))
    assert isinstance(ns.internal_sampler, type(smp))
    assert ns.internal_sampler.model is m                  # survives _new_from_template


def test_reference_bound_with_b200_sampler(dynesty, fake_ops):
    """A foreign Bound (the reference's own MultiEllipsoid, bound='multi') feeding the B200
    rwalk sampler: axes arrive as plain ndarrays and are uploaded per fill."""
    c, b, s = _classes()
    from dynesty_b200 import likelihoods as DL
    from dynesty_b200.pool import B200Pool
    m = DL.gauss_test3d()
    ns = dynesty.NestedSampler(m.loglikelihood, m.prior_transform, 3, nlive=100, bound='multi',
                               sample=s.B200RWalkSampler(model=m, walks=10), pool=B200Pool(16),
                               queue_size=16, rstate=np.random.default_rng(1),
                               use_pool={'prior_transform': False, 'loglikelihood': False})
    ns.run_nested(dlogz=0.5, print_progress=False)
    assert abs(ns.results['logz'][-1] - 3 * (-np.log(20.))) < 5 * ns.results['logzerr'][-1] + 0.1


def test_sampler_requires_model():
    c, b, s = _classes()
    with pytest.raises(ValueError):
        s.B200RWalkSampler(walks=5)


def test_dropin_dynamic_sampler(dynesty, fake_ops):
    """BASELINE C5 shape: DynamicNestedSampler(bound='multi', sample='rslice') re-enters the
    same plug-in path for every batch (dynamicsampler.py:373-390, 1094-1110)."""
    c, b, s = _classes()
    from dynesty_b200 import likelihoods as DL
    from dynesty_b200.pool import B200Pool
    m = DL.shells(2)
    ds = dynesty.DynamicNestedSampler(m.loglikelihood, m.prior_transform, 2, bound=b.B200MultiEllipsoid(2),
                                      sample=s.B200RSliceSampler(model=m, slices=3), pool=B200Pool(16),
                                      queue_size=16, rstate=np.random.default_rng(4),
                                      use_pool={'prior_transform': False, 'loglikelihood': False})
    ds.run_nested(nlive_init=100, nlive_batch=50, maxbatch=2, dlogz_init=0.5, print_progress=False)
    res = ds.results
    assert abs(res['logz'][-1] - (-1.75)) < 5 * res['logzerr'][-1] + 0.15
    assert len(res['batch_nlive']) >= 2


def test_dropin_checkpoint_restore(dynesty, fake_ops, tmp_path):
    """The reference's own checkpointing (Sampler.save -> utils.save_sampler pickles the whole sampler,
    utils.py:2321-2355; tests/test_resume.py) with the B200 bound / sampler / pool inside: the plug-in objects
    must pickle (device handles dropped, re-created lazily) and the restored sampler must keep running."""
    c, b, s = _classes()
    from dynesty_b200 import likelihoods as DL
    from dynesty_b200.pool import B200Pool
    m = DL.gauss_test3d()
    mk = lambda: dynesty.NestedSampler(m.loglikelihood, m.prior_transform, 3, nlive=100, bound=b.B200MultiEllipsoid(3),
                                       sample=s.B200RWalkSampler(model=m, walks=10), pool=B200Pool(16), queue_size=16,
                                       rstate=np.random.default_rng(9),
                                       use_pool={'prior_transform': False, 'loglikelihood': False})
    f = str(tmp_path / 'dyn.save')
    ns = mk()
    ns.run_nested(maxiter=700, dlogz=1e-9, print_progress=False, checkpoint_file=f, add_live=False)
    assert ns.nbound > 1
    ns.save(f)
    r = dynesty.NestedSampler.restore(f, pool=B200Pool(16))
    assert isinstance(r.bound, b.B200MultiEllipsoid) and isinstance(r.internal_sampler, s.B200RWalkSampler)
    assert r.it == ns.it and np.array_equal(r.live_logl, ns.live_logl)
    assert np.array_equal(r.bound.ctrs, ns.bound.ctrs) and r.internal_sampler.scale == ns.internal_sampler.scale
    r.run_nested(dlogz=0.5, print_progress=False, resume=True)
    assert abs(r.results['logz'][-1] - 3 * (-np.log(20.))) < 5 * r.results['logzerr'][-1] + 0.1
    assert r.results["niter"] > 700


def test_pool_size_sets_the_queue(dynesty, fake_ops):
    """utils.py:2358-2381 _parse_pool_queue: without queue_size the Sampler takes it from ``pool.size`` -- the
    number of chains the B200 pool advertises = chains per kernel launch."""
    c, b, s = _classes()
    from dynesty_b200 import likelihoods as DL
    from dynesty_b200.pool import B200Pool
    m = DL.gauss_test3d()
    ns = dynesty.NestedSampler(m.loglikelihood, m.prior_transform, 3, nlive=60, bound=b.B200Ellipsoid(3),
                               sample=s.B200RSliceSampler(model=m, slices=2), pool=B200Pool(24),
                               rstate=np.random.default_rng(3),
                               use_pool={'prior_transform': False, 'loglikelihood': False})
    assert ns.queue_size == 24
    ns.run_nested(maxiter=300, dlogz=1e-9, print_progress=False, add_live=False)
    assert ns.internal_sampler.last_batch is not None and len(ns.internal_sampler.last_batch['logl']) == 24


@pytest.mark.parametrize('kind,sample', [('balls', 'unif'), ('cubes', 'unif'), ('balls', 'rwalk')])
def test_dropin_friends(dynesty, fake_ops, kind, sample):
    """B200RadFriends / B200SupFriends under the unmodified dynesty.NestedSampler: ``need_centers`` makes the Sampler
    assign its live points to ``bound.ctrs`` (sampler.py:479-482); ``contains`` of a start point (a centre) is True."""
    c, b, s = _classes()
    from dynesty_b200 import likelihoods as DL
    from dynesty_b200.pool import B200Pool
    from dynesty import bounding as RB
    m = DL.gauss_test3d()
    bnd = (b.B200RadFriends if kind == 'balls' else b.B200SupFriends)(3)
    assert isinstance(bnd, RB.Bound) and bnd.need_centers
    smp = s.B200UniformSampler(model=m) if sample == 'unif' else s.B200RWalkSampler(model=m, walks=10)
    ns = dynesty.NestedSampler(m.loglikelihood, m.prior_transform, 3, nlive=80, bound=bnd, sample=smp,
                               pool=B200Pool(16), queue_size=16, rstate=np.random.default_rng(3), bootstrap=0,
                               use_pool={'prior_transform': False, 'loglikelihood': False})
    ns.run_nested(dlogz=0.5, print_progress=False)
    res = ns.results
    assert abs(res['logz'][-1] - 3 * (-np.log(20.))) < 5 * res['logzerr'][-1] + 0.1
    assert ns.nbound > 1 and isinstance(ns.bound, type(bnd)) and ns.bound.ctrs is ns.live_u
