"""Generate tests/golden/*.npz by running the UNMODIFIED reference.

TEST INFRASTRUCTURE.  Needs the reference: a dynesty checkout or its copy oracle/_ref
(oracle/refshim.py):

    python -m oracle.make_golden [bounding friends chains dynamic]    (default: all)

Every output array below is produced by the reference's own functions
(dynesty 3.0.0+ @ 99451618, imported through oracle/refshim.py); stochastic
ones are driven by ``oracle.philox.ScriptedGenerator`` so that the reference
consumes the B2N Philox stream.  The oracle restatement (oracle/*.py) and the
CUDA path are both tested against these files.
"""
import os
import warnings
import numpy as np

from . import refshim, philox, likelihoods as L

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                   'tests', 'golden')
SEED = 56432          # tests/utils.py:12-20 convention of the reference


def cloud_gauss(rng, npts, n, spread=0.04, rho=0.4):
    """Live-point-like cloud in the unit cube: correlated Gaussian blob."""
    C = np.full((n, n), rho)
    np.fill_diagonal(C, 1.0)
    Lc = np.linalg.cholesky(C)
    return 0.5 + spread * rng.standard_normal((npts, n)) @ Lc.T


def cloud_clusters(rng, npts, n, k, spread=0.01):
    ctr = 0.15 + 0.7 * rng.random((k, n))
    lab = rng.integers(k, size=npts)
    return ctr[lab] + spread * rng.standard_normal((npts, n)), lab


def ell_dict(prefix, e):
    return {prefix + 'ctr': e.ctr, prefix + 'cov': e.cov, prefix + 'am': e.am,
            prefix + 'axes': e.axes, prefix + 'axlens': e.axlens,
            prefix + 'logvol': np.float64(e.logvol)}


def gen_bounding(B):
    rng = np.random.default_rng(SEED)
    out = {}
    # (1) single bounding ellipsoids on seeded clouds  (bounding.py:1387-1461)
    clouds = {
        'g20': cloud_gauss(rng, 600, 20),
        'g3': cloud_gauss(rng, 200, 3, spread=0.1, rho=0.95),
        'g50': cloud_gauss(rng, 400, 50, spread=0.02),
        'few': cloud_gauss(rng, 5, 4),                 # npoints ~ ndim
    }
    # rank-deficient data (tests/test_ellipsoid.py:258-264 test_bounding_crazy)
    x = rng.random(100)
    clouds['rank1'] = 0.5 + (x[:, None] - 0.5) * np.ones((1, 10)) * 0.3
    # strongly ill-conditioned (condition number > 1e12 -> ladder branch 1)
    ill = cloud_gauss(rng, 300, 6, spread=0.05, rho=0.0)
    ill[:, 0] = 0.5 + 1e-9 * (ill[:, 0] - 0.5)
    clouds['illcond'] = ill
    for name, pts in clouds.items():
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            e = B.bounding_ellipsoid(pts)
        out['be_%s_points' % name] = pts
        out.update(ell_dict('be_%s_' % name, e))
    # (2) improve_covar_mat on the reference's own test inputs
    #     (tests/test_ellipsoid.py:242-255)
    for name, mat in {
            'zero': np.zeros((4, 4)),
            'rank1': np.outer(np.arange(1., 6.), np.arange(1., 6.)),
            'neg': np.diag([1., -1., 2.]),
            'good': np.cov(cloud_gauss(rng, 50, 5), rowvar=False)}.items():
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            good, cov, am, axes = B.improve_covar_mat(mat)
        out['icm_%s_in' % name] = mat
        out['icm_%s_good' % name] = np.bool_(good)
        out['icm_%s_cov' % name] = cov
        out['icm_%s_am' % name] = am
        out['icm_%s_axes' % name] = axes
    # (3) scale_to_logvol: isotropic branch and capped branch (bounding.py:242-276)
    e = B.bounding_ellipsoid(clouds['g20'])
    out.update(ell_dict('stl_in_', e))
    import copy
    for name, dlv in {'iso': 0.223, 'cap': 60.0, 'shrink': -1.5}.items():
        e2 = copy.deepcopy(e)
        e2.scale_to_logvol(e.logvol + dlv)
        out['stl_%s_dlv' % name] = np.float64(dlv)
        out.update(ell_dict('stl_%s_' % name, e2))
    # (4) kmeans2 as the reference calls it (bounding.py:1510-1514)
    from scipy.cluster.vq import kmeans2
    pts, _ = cloud_clusters(rng, 500, 5, 2, spread=0.05)
    e = B.bounding_ellipsoid(pts)
    p1, p2 = e.major_axis_endpoints()
    start = np.vstack((p1, p2))
    scale = pts.std(axis=0)[None, :]
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        cb, lab = kmeans2(pts / scale, k=start / scale, iter=10, minit='matrix',
                          check_finite=False)
    out['km_points'] = pts
    out['km_start'] = start
    out['km_scale'] = scale
    out['km_code'] = cb
    out['km_labels'] = lab.astype(np.int32)
    np.savez_compressed(os.path.join(OUT, 'bounding.npz'), **out)

    # (5) multi-ellipsoid decomposition (bounding.py:632-686, 1464-1563)
    out = {}
    cases = {
        'c8': cloud_clusters(rng, 1600, 10, 8)[0],
        'c2': cloud_clusters(rng, 400, 5, 2, spread=0.03)[0],
        'blob': cloud_gauss(rng, 500, 8),
        'ring': None,
    }
    t = rng.random(1200) * 2 * np.pi
    cases['ring'] = 0.5 + 0.3 * np.stack([np.cos(t), np.sin(t)], 1) + \
        0.01 * rng.standard_normal((1200, 2))
    for name, pts in cases.items():
        n = pts.shape[1]
        me = B.MultiEllipsoid(n)
        me.update(pts)
        out['me_%s_points' % name] = pts
        out['me_%s_ctrs' % name] = me.ctrs
        out['me_%s_covs' % name] = me.covs
        out['me_%s_ams' % name] = me.ams
        out['me_%s_axes' % name] = np.array([e.axes for e in me.ells])
        out['me_%s_logvols' % name] = me.logvol_ells
        out['me_%s_logvol' % name] = np.float64(me.logvol)
        # membership of query points (bounding.py:502-523), strict <
        q = np.vstack([pts[:300], rng.random((700, n))])
        d = q[:, None, :] - me.ctrs[None]
        mask = np.array([[i in me.within(x) for i in range(me.nells)] for x in q])
        out['me_%s_query' % name] = q
        out['me_%s_mask' % name] = mask
        out['me_%s_contains' % name] = np.array([me.contains(x) for x in q])
        # enlarge as Sampler.update_bound does (sampler.py:506-508)
        me.scale_to_logvol(me.logvol + np.log(1.25))
        out['me_%s_enl_ams' % name] = me.ams
        out['me_%s_enl_axes' % name] = np.array([e.axes for e in me.ells])
        out['me_%s_enl_logvols' % name] = me.logvol_ells
    # (6) bootstrap expansion factors (bounding.py:1593-1648), scripted integers
    pts = cases['c2']
    for multi in (False, True):
        exps = []
        for rep in range(4):
            g = philox.ScriptedGenerator(SEED, 1000 + rep)
            exps.append(B._ellipsoid_bootstrap_expand((multi, pts, g)))
        out['boot_%d_expand' % multi] = np.array(exps)
    np.savez_compressed(os.path.join(OUT, 'multi.npz'), **out)


def run_ref_chains(IS, cls, model, u0s, loglstar, axes, scale, kwargs, chain0):
    """Drive the reference's static ``sample`` (internal_samplers.py:505, 594,
    746) once per start point with a scripted generator."""
    res = []
    for i, u0 in enumerate(u0s):
        g = philox.ScriptedGenerator(SEED, chain0 + i)
        ax = axes[i] if isinstance(axes, list) else axes
        args = IS.SamplerArgument(u=u0.copy(), loglstar=loglstar, axes=ax,
                                  scale=scale,
                                  prior_transform=model.prior_transform,
                                  loglikelihood=lambda v: float(model.loglike(v)),
                                  rseed=g, kwargs=kwargs)
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            r = cls.sample(args)
        res.append((r, g.tick))
    return res


def pack_chain(prefix, res, keys):
    d = {prefix + 'u': np.array([r.u for r, _ in res]),
         prefix + 'v': np.array([r.v for r, _ in res]),
         prefix + 'logl': np.array([r.logl for r, _ in res]),
         prefix + 'ncall': np.array([r.ncalls for r, _ in res], dtype=np.int64),
         prefix + 'ticks': np.array([t for _, t in res], dtype=np.int64)}
    for k in keys:
        d[prefix + k] = np.array([r.tuning_info[k] for r, _ in res], dtype=np.int64)
    return d


def starts_above(model, pts, frac):
    logl = model.loglike(model.prior_transform(pts))
    loglstar = float(np.quantile(logl, frac))
    return pts[logl > loglstar], loglstar


def gen_chains(B, IS):
    rng = np.random.default_rng(SEED + 1)
    out = {}
    meta = {}

    def add_rwalk(name, model, pts, ncdim, walks, scale, nchain, periodic=None,
                  reflective=None, chain0=0):
        n = model.ndim
        e = B.bounding_ellipsoid(pts[:, :ncdim])
        st, loglstar = starts_above(model, pts, 0.3)
        st = st[:nchain]
        nonb = None
        if periodic is not None or reflective is not None:
            nonb = np.ones(n, dtype=bool)
            if periodic is not None:
                nonb[periodic] = False
            if reflective is not None:
                nonb[reflective] = False
        kw = dict(walks=walks, ncdim=ncdim, nonbounded=nonb, periodic=periodic,
                  reflective=reflective)
        res = run_ref_chains(IS, IS.RWalkSampler, model, st, loglstar, e.axes,
                             scale, kw, chain0)
        p = 'rwalk_%s_' % name
        out.update(pack_chain(p, res, ['accept', 'reject']))
        out[p + 'u0'] = st
        out[p + 'axes'] = e.axes
        out[p + 'loglstar'] = np.float64(loglstar)
        out[p + 'scale'] = np.float64(scale)
        out[p + 'walks'] = np.int64(walks)
        out[p + 'ncdim'] = np.int64(ncdim)
        out[p + 'chain0'] = np.int64(chain0)
        out[p + 'periodic'] = np.array([] if periodic is None else periodic, dtype=np.int64)
        out[p + 'reflective'] = np.array([] if reflective is None else reflective, dtype=np.int64)

    m6 = L.gauss_corr(6, 0.4, 5.)
    add_rwalk('g6', m6, cloud_gauss(rng, 300, 6, spread=0.06), 6, 25, 0.8, 24, chain0=100)
    add_rwalk('g6nc', m6, cloud_gauss(rng, 300, 6, spread=0.06), 4, 25, 0.8, 24,
              periodic=[1], reflective=[2], chain0=200)
    # near the cube wall so that wrap / reflect / out-of-cube rejects all occur
    wall = cloud_gauss(rng, 300, 6, spread=0.06)
    wall[:, :3] -= 0.42
    wall = np.abs(wall)
    m6w = L.Model(6, L.PRIOR_UNIFORM, L.LIKE_GAUSS_PREC, lo=np.full(6, -5.),
                  width=np.full(6, 10.), mean=np.r_[-4.2, -4.2, -4.2, 0, 0, 0.],
                  prec=m6.p['prec'], lnorm=m6.p['lnorm'])
    add_rwalk('wall', m6w, wall, 6, 30, 1.5, 24, periodic=[0], reflective=[1],
              chain0=300)
    m50 = L.gauss_corr(50, 0.4, 5.)
    add_rwalk('g50', m50, cloud_gauss(rng, 400, 50, spread=0.02), 50, 70, 0.35, 12,
              chain0=400)
    m200 = L.iid_normal_ppf(200)
    pts200 = 0.5 + 0.03 * rng.standard_normal((600, 200))
    add_rwalk('n200', m200, pts200, 200, 12, 0.2, 4, chain0=500)

    def add_slice(kind, name, model, pts, slices, scale, nchain, doubling, chain0):
        e = B.bounding_ellipsoid(pts)
        st, loglstar = starts_above(model, pts, 0.3)
        st = st[:nchain]
        kw = dict(slices=slices, nonbounded=None, periodic=None, reflective=None)
        if doubling:
            kw['slice_doubling'] = True
        cls = IS.RSliceSampler if kind == 'rslice' else IS.SliceSampler
        res = run_ref_chains(IS, cls, model, st, loglstar, e.axes, scale, kw, chain0)
        p = '%s_%s_' % (kind, name)
        out.update(pack_chain(p, res, ['n_expand', 'n_contract']))
        out[p + 'u0'] = st
        out[p + 'axes'] = e.axes
        out[p + 'loglstar'] = np.float64(loglstar)
        out[p + 'scale'] = np.float64(scale)
        out[p + 'slices'] = np.int64(slices)
        out[p + 'doubling'] = np.bool_(doubling)
        out[p + 'chain0'] = np.int64(chain0)

    egg = L.eggbox(5)
    pe = rng.random((400, 5))
    sh = L.shells(4)
    ps = rng.random((3000, 4))
    ps = ps[np.argsort(sh.loglike(sh.prior_transform(ps)))[-400:]]
    g4 = L.gauss_corr(4, 0.6, 5.)
    pg = cloud_gauss(rng, 300, 4, spread=0.07, rho=0.6)
    for dbl in (False, True):
        tag = 'dbl' if dbl else 'std'
        add_slice('rslice', 'egg_' + tag, egg, pe, 6, 0.5, 16, dbl, 600 + 50 * dbl)
        add_slice('rslice', 'shell_' + tag, sh, ps, 6, 0.3, 16, dbl, 700 + 50 * dbl)
        add_slice('rslice', 'g4_' + tag, g4, pg, 7, 1.0, 16, dbl, 800 + 50 * dbl)
        add_slice('slice', 'g4_' + tag, g4, pg, 3, 1.0, 16, dbl, 900 + 50 * dbl)
        add_slice('slice', 'egg_' + tag, egg, pe, 2, 0.5, 16, dbl, 1000 + 50 * dbl)

    # uniform sampling within the bound (internal_samplers.py:243-340)
    def add_unif(name, model, pts, ncdim, nchain, chain0, frac=0.5):
        n = model.ndim
        me = B.MultiEllipsoid(ncdim)
        me.update(pts[:, :ncdim])
        me.scale_to_logvol(me.logvol + np.log(1.25))
        logl = model.loglike(model.prior_transform(pts))
        loglstar = float(np.quantile(logl, frac))
        kw = dict(bound=me, ndim=n, n_cluster=ncdim, nonbounded=None)
        res = run_ref_chains(IS, IS.UniformBoundSampler, model,
                             [pts[0]] * nchain, loglstar, me.ells[0].axes, 1.0, kw,
                             chain0)
        p = 'unif_%s_' % name
        d = pack_chain(p, res, [])
        out.update(d)
        out[p + 'ctrs'] = me.ctrs
        out[p + 'ams'] = me.ams
        out[p + 'axes'] = np.array([e.axes for e in me.ells])
        out[p + 'logvols'] = me.logvol_ells
        out[p + 'loglstar'] = np.float64(loglstar)
        out[p + 'chain0'] = np.int64(chain0)
        out[p + 'ndim'] = np.int64(n)

    g3 = L.gauss_test3d()
    p3 = cloud_gauss(rng, 300, 3, spread=0.05, rho=0.95)
    p3 += np.linspace(-1, 1, 3) / 20.
    add_unif('g3', g3, p3, 3, 24, 1200)
    add_unif('g3nc', g3, p3, 2, 24, 1300)
    # two overlapping clusters -> K >= 2 with q > 1 rejections
    sh2 = L.shells(2)
    pp = rng.random((20000, 2))
    pp = pp[np.argsort(sh2.loglike(sh2.prior_transform(pp)))[-600:]]
    add_unif('shell2', sh2, pp, 2, 24, 1400, frac=0.2)
    # the sampler of the phase before the first bound: UnitCubeSampler.sample (internal_samplers.py:343-441),
    # replayed on the Philox stream like the others (added in round 2, after every earlier fixture)
    uc_thr = -20.0
    res = run_ref_chains(IS, IS.UnitCubeSampler, g3, [p3[0]] * 32, uc_thr, np.eye(3), 1.0, dict(ndim=3), 1500)
    out.update(pack_chain('uc_', res, []))
    out['uc_loglstar'], out['uc_seed'], out['uc_chain0'] = np.float64(uc_thr), np.int64(SEED), np.int64(1500)
    np.savez_compressed(os.path.join(OUT, 'chains.npz'), **out)
    return out


def gen_friends(B):
    """RadFriends / SupFriends (bounding.py:734-1263): two successive updates (the second clusters with the
    first one's am), leave-one-out and bootstrap radii, overlap counts, scripted draws."""
    rng = np.random.default_rng(SEED + 7)
    out = {}
    clouds = {'blob': cloud_gauss(rng, 160, 4, spread=0.05),
              'two': np.concatenate([0.25 + 0.02 * rng.standard_normal((90, 3)),
                                     0.75 + 0.02 * rng.standard_normal((90, 3))])}
    for cname, pts in clouds.items():
        n = pts.shape[1]
        for kind, cls in (('balls', B.RadFriends), ('cubes', B.SupFriends)):
            p = 'fr_%s_%s_' % (cname, kind)
            out[p + 'points'] = pts
            b = cls(n)
            for rep in (1, 2):
                b.update(pts if rep == 1 else pts[::-1][:len(pts) - 10], rstate=np.random.default_rng(1), bootstrap=0)
                b.ctrs = pts if rep == 1 else pts[::-1][:len(pts) - 10]
                q = p + 'u%d_' % rep
                out[q + 'cov'], out[q + 'am'], out[q + 'axes'] = b.cov.copy(), b.am.copy(), np.real(b.axes).copy()
                out[q + 'axes_inv'], out[q + 'logvol'] = np.real(b.axes_inv).copy(), np.float64(b.logvol)
                # the Sampler enlarges after every update (sampler.py:506-508).  Without it the pair that
                # defines the leave-one-out radius sits at Mahalanobis distance exactly 1 -- the clustering
                # threshold of the NEXT update -- and the partition would hinge on the last bit
                b.scale_to_logvol(b.logvol + np.log(1.25))
            xs = np.concatenate([pts[:20] + 0.01 * rng.standard_normal((20, n)), rng.random((20, n))])
            out[p + 'query'] = xs
            out[p + 'overlap'] = np.array([b.overlap(x) for x in xs])
            out[p + 'contains'] = np.array([b.contains(x) for x in xs])
            # radii helpers on the decorrelated points (bounding.py:1651-1705)
            pt = np.dot(b.ctrs, np.real(b.axes_inv))
            out[p + 'loo'] = B._friends_leaveoneout_radius(pt, kind)
            brad = []
            for r in range(3):
                g = philox.ScriptedGenerator(SEED, 400 + r)
                brad.append(B._friends_bootstrap_radius((pt, kind, g)))
            out[p + 'boot'] = np.array(brad)
            # scripted draws: sample() and sample(return_q=True)
            xs1, qs = [], []
            for c in range(30):
                g = philox.ScriptedGenerator(SEED, 500 + c)
                xs1.append(b.sample(rstate=g))
                x, qq = b.sample(rstate=philox.ScriptedGenerator(SEED, 600 + c), return_q=True)
                xs1.append(x)
                qs.append(qq)
            out[p + 'draws'] = np.array(xs1)
            out[p + 'draw_q'] = np.array(qs)
            lv0 = b.logvol
            b.scale_to_logvol(lv0 + 0.3)
            out[p + 'scaled_am'], out[p + 'scaled_axes'] = b.am.copy(), np.real(b.axes).copy()
    np.savez_compressed(os.path.join(OUT, 'friends.npz'), **out)
    return out


def gen_dynamic():
    """dynamic.npz: the reference's own dynamicsampler.weight_function / compute_weights and
    utils.compute_integrals evaluated on the results of one device-loop run (3-D Gaussian, nlive 100, multi /
    rwalk, rounds of 10) made on the oracle backend (tests/fake_backend.py).  The inputs are stored with the
    outputs, so tests/test_dynamic.py and tests/test_oracle_nsloop.py compare with the reference without it."""
    import sys
    import types
    import pytest
    sys.path.insert(0, os.path.dirname(OUT))          # tests/: the oracle backend
    import fake_backend
    from dynesty import dynamicsampler as RD, utils as RU
    from dynesty_b200 import nested, likelihoods as DL
    mp = pytest.MonkeyPatch()
    try:
        fake_backend.install(mp)
        s = nested.NestedSampler(DL.gauss_test3d(), nlive=100, bound='multi', sample='rwalk', walks=8, seed=2)
        res = s.run_nested(dlogz=0.1, loop='device', batch=10)
    finally:
        mp.undo()
    out = {k: np.asarray(getattr(res, k)) for k in ('logl', 'logz', 'logvol', 'logwt', 'samples_n')}
    R = types.SimpleNamespace(**out)
    out['weight_bounds'] = np.array([RD.weight_function(R, a) for a in WEIGHT_ARGS], dtype=float)
    out['zweight'], out['pweight'] = RD.compute_weights(R)
    out['integrals_logwt'], out['integrals_logz'] = RU.compute_integrals(logl=out['logl'], logvol=out['logvol'])[:2]
    np.savez_compressed(os.path.join(OUT, 'dynamic.npz'), **out)
    return out


# the weight_function arguments of dynamic.npz's 'weight_bounds', row by row (None = the defaults)
WEIGHT_ARGS = (None, dict(pfrac=0.0), dict(pfrac=1.0, maxfrac=0.5, pad=3))


FIXTURES = ('bounding', 'friends', 'chains', 'dynamic')


def main(which=FIXTURES):
    os.makedirs(OUT, exist_ok=True)
    refshim.import_reference()
    from dynesty import bounding as B, internal_samplers as IS
    if 'bounding' in which:
        gen_bounding(B)
    if 'friends' in which:
        gen_friends(B)
    if 'chains' in which:
        out = gen_chains(B, IS)
        ku = [k for k in out if k.endswith('_logvols') and k.startswith('unif')]
        print({k: len(out[k]) for k in ku})
    if 'dynamic' in which:
        gen_dynamic()
    print('wrote', OUT, {k: os.path.getsize(os.path.join(OUT, k))
                         for k in sorted(os.listdir(OUT))})


if __name__ == '__main__':
    import sys
    main(sys.argv[1:] or FIXTURES)
