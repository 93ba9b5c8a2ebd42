"""CPU tier: dynesty_b200/dynamic.py -- the dynamic sampler whose baseline and batches are device rounds.  The merge is
checked against a literal restatement of the reference's ``combine_runs`` loop (dynamicsampler.py:1500-1560), the
weight function against stored outputs of the reference's own ``weight_function``, and a whole run
against the analytic evidence on the oracle backend."""
import os

import numpy as np
import pytest

from dynesty_b200 import dynamic as D, likelihoods as DL
from oracle import make_golden


def _loop_merge(ls, ns, ln, nn, logl_min):
    """combine_runs' stepping loop, literally."""
    out_l, out_n, src = [], [], []
    i = j = 0
    logl_s, logl_n = ls[0], ln[0]
    nlive_s, nlive_n = ns[0], nn[0]
    for _ in range(len(ls) + len(ln)):
        nlive = nlive_s + nlive_n if logl_s > logl_min else nlive_s
        if logl_s <= logl_n:
            out_l.append(ls[i]); src.append(0); i += 1
        else:
            out_l.append(ln[j]); src.append(1); j += 1
        out_n.append(nlive)
        logl_s, nlive_s = (ls[i], ns[i]) if i < len(ls) else (np.inf, 0)
        logl_n, nlive_n = (ln[j], nn[j]) if j < len(ln) else (np.inf, 0)
    return np.array(out_l), np.array(out_n), np.array(src)


@pytest.mark.parametrize('seed', [0, 1, 2])
def test_merge_two_equals_the_reference_loop(seed):
    rng = np.random.default_rng(seed)
    ls = np.sort(rng.normal(size=60))
    ns = np.r_[np.full(40, 20), 20 - np.arange(20)]                    # constant, then the add_live tail
    lo = ls[15]
    ln = np.sort(np.r_[rng.uniform(lo, ls[-1] + 1, size=35), ls[30]])  # one exact tie with a saved point
    nn = np.r_[np.tile(12 - np.arange(4), 6), 12 - np.arange(12)]      # rounds of 4 removals, then the tail
    rec_s = dict(logl=ls, n=ns, tag=np.zeros(60))
    rec_n = dict(logl=ln, n=nn, tag=np.ones(36))
    m = D.merge_two(rec_s, rec_n, lo)
    el, en, src = _loop_merge(ls, ns, ln, nn, lo)
    assert np.array_equal(m['logl'], el) and np.array_equal(m['n'], en) and np.array_equal(m['tag'], src)
    assert np.all(np.diff(m['logl']) >= 0)


def test_weight_function_matches_reference():
    """The reference's own weight_function / compute_weights on the results of a device-loop run (oracle backend),
    stored with those results in tests/golden/dynamic.npz by oracle/make_golden.py."""
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'dynamic.npz'))
    res = {k: g[k] for k in ('logl', 'logz', 'logvol', 'logwt', 'samples_n')}
    for args, a in zip(make_golden.WEIGHT_ARGS, g['weight_bounds']):
        b = D.weight_function(res, args)
        assert a[0] == b[0] and a[1] == b[1]
    za, pa = g['zweight'], g['pweight']
    zb, pb = D.compute_weights(res)
    np.testing.assert_allclose(za, zb, rtol=1e-9)
    np.testing.assert_allclose(pa, pb, rtol=1e-12)


def test_dynamic_run_on_the_oracle_backend(fake_ops):
    m = DL.gauss_test3d()
    d = D.DynamicNestedSampler(m, nlive=80, bound='multi', sample='rwalk', walks=10, seed=4)
    r0 = d.sample_initial(dlogz=0.5, round_size=8)
    n0 = r0.niter
    res = d.run_nested(nlive_batch=60, maxbatch=2, n_effective=1e9, round_size=6)
    assert d.batch == 2 and res.niter > n0 and len(res.batch_bounds) == 3
    assert np.all(np.diff(res.logl) >= 0) and np.all(np.diff(res.logvol) < 0)
    assert set(np.unique(res.samples_batch)) == {0, 1, 2}
    lo, hi = res.batch_bounds[1]
    inside = (res.logl > lo) & (res.logl < min(hi, res.logl[res.samples_batch == 1].max()))
    assert res.samples_n[inside].max() > 80                         # the two runs' live points add up where they overlap
    truth = 3 * (-np.log(20.))
    assert abs(res.logz[-1] - truth) < 4 * res.logzerr[-1] + 0.1
    w = np.exp(res.logwt - res.logz[-1])
    mean = (w / w.sum()) @ res.samples
    assert np.all(np.abs(mean - np.linspace(-1, 1, 3)) < 0.4)
    assert D.n_effective_of(res) > D.n_effective(r0.logwt)
