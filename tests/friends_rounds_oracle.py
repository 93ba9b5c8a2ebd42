"""TEST-ONLY restatement of the device rounds with a RadFriends / SupFriends bound (friends mode of csrc/b2n_ns.cu),
built on the rounds' oracle ``oracle.nsloop.BatchNS`` and the friends oracle ``oracle.friends.Friends``.

What differs from the ellipsoid rounds (reference py/dynesty/):
  chain samplers   the common axes of the bound (get_random_axes, bounding.py:995-997 / 1262-1264) and no contains test:
                   a start point is a live point, hence a centre (distance 0), so sampler.py:485-489 cannot fire.  Both
                   follow from handing BatchNS a one-"ellipsoid" view of the bound whose metric is zero (every point
                   inside).
  uniform sampler  every chain of a round draws with ``Friends.sample`` (bounding.py:797-831 / 1065-1100) around the live
                   set as it stands at the start of the round (sampler.py:479-482: bound.ctrs = live_u), then the
                   unit-cube test, the prior transform and the likelihood (UniformBoundSampler, internal_samplers.py:
                   243-340).  Draw events per try: the offset, the centre uniform when N > 1, the 1/q uniform unless q == 1.
  bootstrap        realisation b of a device update made at round r resamples with the B2N chain
                   FRIENDS_BOOT_CHAIN + (r << 8) + b (b2n_ns_update_friends, include/b200nest.h).
"""
import numpy as np

from oracle import nsloop, philox, samplers as OS
from oracle.friends import Friends

FRIENDS_BOOT_CHAIN = 0x6000000000000000


def friends_boot_idxs(seed, round_, nboot, npoints):
    """Resample indices of the `nboot` bootstrap realisations of a friends update made at round `round_`: one uniform
    vector event of the chain FRIENDS_BOOT_CHAIN + (round_ << 8) + b each, for ``Friends.update(bootstrap_idxs=...)``.
    None when nboot == 0 (leave-one-out radius)."""
    if not nboot:
        return None
    return [philox.ChainStream(seed, FRIENDS_BOOT_CHAIN + (int(round_) << 8) + b).integers(npoints, npoints)
            for b in range(int(nboot))]


def friends_unif_chain(loglstar, bound, model, stream, nonbounded=None, max_tries=10**7):
    """UniformBoundSampler.sample with a Friends bound: bound draws until one inside the unit cube has logl > loglstar."""
    ncall = 0
    for _ in range(max_tries):
        x = bound.sample(stream)
        if not OS.unitcheck(x, nonbounded):                      # internal_samplers.py:314
            continue
        v = model.prior_transform(x)
        logl = float(model.loglike(v))
        ncall += 1
        if logl > loglstar:
            return dict(u=x, v=v, logl=logl, ncall=ncall, ticks=stream.tick)
    raise RuntimeError("friends_unif_chain: no point found")


def chain_view(f):
    """The bound as the chain samplers of BatchNS see it: one "ellipsoid" with the common axes and a zero metric."""
    n = f.ndim
    return dict(ctrs=np.zeros((1, n)), ams=np.zeros((1, n, n)), axes=np.asarray(f.axes)[None],
                logvols=np.array([float(f.logvol)]), strict=True)


class FriendsBatchNS(nsloop.BatchNS):
    """BatchNS whose bound is an ``oracle.friends.Friends`` (``friends``); same constructor otherwise."""

    def __init__(self, *a, friends=None, **kw):
        super().__init__(*a, **kw)
        self.friends = None
        if friends is not None:
            self.use(friends)

    def use(self, f):
        self.friends = f
        self.bound = chain_view(f)

    def bound_updated(self, bound=None):
        if isinstance(bound, Friends):
            self.use(bound)
            bound = None
        super().bound_updated(bound)

    def _step_unif(self, order, sl, thr):
        if self.friends is None:
            return super()._step_unif(order, sl, thr)
        f = self.friends
        f.ctrs = self.live_u.copy()
        out = [friends_unif_chain(thr, f, self.model,
                                  philox.ChainStream(self.seed, self.chain0 + self.round * self.K + c), nonbounded=self.nb)
               for c in range(self.K)]
        self._commit(order, sl, thr, out)
        self.last = dict(thr=thr)
        if self.ncall >= self.ncall_last_update + self.update_interval:
            self.need_bound = 1
        return True
