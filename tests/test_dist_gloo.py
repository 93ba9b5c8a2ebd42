"""CPU tier: the N>1 path (chains of a queue fill sharded over ranks + all-gather) with
world_size=2 on the gloo backend.  Kernels are replaced by the oracle-backed stand-in
(tests/fake_backend.py); what is pinned is that the sharded run is IDENTICAL to the
single-rank run (global chain ids -> same Philox streams) and that every rank ends with the
same state."""
import os
import socket
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _run(rank, world, port, outdir, sample='rwalk', patch=None):
    """One rank of the run.  `patch`: the calling test's monkeypatch when the rank runs inside the pytest process,
    so that the stand-in backend and the environment are restored when the test ends (later tests in the same
    session, the GPU ones included, must see the real library)."""
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    patch = patch or pytest.MonkeyPatch()
    for k, v in dict(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world)).items():
        patch.setenv(k, v)
    import torch.distributed as dist
    import fake_backend
    from dynesty_b200 import ops, likelihoods as DL, nested
    from dynesty_b200.dist import Comm

    fake_backend.install(patch)
    comm = None
    if world > 1:
        dist.init_process_group('gloo', rank=rank, world_size=world)
        comm = Comm()
    m = DL.gauss_test3d()
    s = nested.NestedSampler(m, nlive=60, bound='multi', sample=sample, walks=8, slices=3, queue_size=20, seed=5,
                             comm=comm)
    res = s.run_nested(dlogz=None, maxiter=250)
    np.savez(os.path.join(outdir, '%s_r%d_w%d.npz' % (sample, rank, world)), logz=res.logz, logl=res.logl,
             samples=res.samples, ncall=res.ncall)
    if world > 1:
        dist.destroy_process_group()


@pytest.mark.parametrize('sample', ['rwalk', 'rslice', 'unif'])
def test_sharded_run_matches_single_rank(tmp_path, monkeypatch, sample):
    """rslice / unif fills return an unsigned `flags` array: the all-gather must carry it (ADVICE r1)."""
    import torch.multiprocessing as mp
    _run(0, 1, 0, str(tmp_path), sample, monkeypatch)
    port = _free_port()
    mp.spawn(_run, args=(2, port, str(tmp_path), sample), nprocs=2, join=True)
    a = np.load(tmp_path / ('%s_r0_w1.npz' % sample))
    b0 = np.load(tmp_path / ('%s_r0_w2.npz' % sample))
    b1 = np.load(tmp_path / ('%s_r1_w2.npz' % sample))
    for k in ('logz', 'logl', 'samples', 'ncall'):
        assert np.array_equal(b0[k], b1[k])            # replicated host state
        assert np.array_equal(a[k], b0[k])             # sharding does not change the run


def test_comm_shard_ranges():
    from dynesty_b200.dist import Comm
    c = Comm.__new__(Comm)
    c.world, c.rank = 4, 2
    assert c.shard(20) == (10, 15)
    with pytest.raises(AssertionError):
        c.shard(18)


def _run_sharded_bound(rank, world, port, outdir):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import torch.distributed as dist
    import fake_backend
    from dynesty_b200 import bounding as B
    from dynesty_b200.dist import Comm

    class MP:
        def setattr(self, obj, name, val):
            setattr(obj, name, val)
    fake_backend.install(MP())
    dist.init_process_group('gloo', rank=rank, world_size=world)
    comm = Comm()
    rng = np.random.default_rng(11)
    pts = 0.5 + 0.05 * rng.standard_normal((301, 7)) @ np.diag(np.linspace(0.3, 2, 7))
    lo, hi = (len(pts) * rank) // world, (len(pts) * (rank + 1)) // world
    b = B.B200Ellipsoid(7)
    b.update_sharded(pts[lo:hi], comm)
    np.savez(os.path.join(outdir, 'sb_r%d.npz' % rank), ctr=b.ctr, cov=b.cov, am=b.am, logvol=b.logvol, pts=pts)
    dist.destroy_process_group()


def test_sharded_bound_update_matches_unsharded(tmp_path):
    """SURVEY 8e for bound='single': rows of the live set sharded over 2 ranks, all-reduce of (count, sum x, scatter)
    and of max delta^T am delta -> the SAME ellipsoid as bounding_ellipsoid of all rows, identical on every rank."""
    import torch.multiprocessing as mp
    from oracle import bounding as OB
    port = _free_port()
    mp.spawn(_run_sharded_bound, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    a, b = np.load(tmp_path / 'sb_r0.npz'), np.load(tmp_path / 'sb_r1.npz')
    for k in ('ctr', 'cov', 'am', 'logvol'):
        assert np.array_equal(a[k], b[k])
    e = OB.bounding_ellipsoid(a['pts'])
    np.testing.assert_allclose(a['ctr'], e.ctr, rtol=1e-12)
    np.testing.assert_allclose(a['cov'], e.cov, rtol=1e-9, atol=1e-15)
    np.testing.assert_allclose(a['am'], e.am, rtol=1e-7)
    assert abs(float(a['logvol']) - e.logvol) < 1e-8
