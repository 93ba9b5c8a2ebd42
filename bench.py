#!/usr/bin/env python
"""bench.py -- proposals/sec of the bounding-and-proposal hot path on B200.

    python bench.py --gpus N --steps K --warmup W            (N>1: under torchrun)
    python bench.py --impl reference --gpus N --steps K --warmup W

A *step* is one pass of the hot path over one batch: one ``_fill_queue`` of the nested
sampler = propose `Q` start points + run `Q` random-walk chains of `walks` proposals each
inside ONE kernel against the resident multi-ellipsoid bound, at a fixed likelihood
threshold (reference sampler.py:676-717 -> internal_samplers.py:866-986).

Workload (BASELINE.json configs[1], "C2"): 50-D correlated Gaussian (rho 0.4, prior
U(-5,5)^50), nlive=2000, bound='multi', sample='rwalk' (walks = ndim+20 = 70), queue of
Q = nlive chains per step, synthetic mid-run live-point state (see make_state).

value  : proposals/s with inputs resident in HBM (device pointers, CUDA events per step).
e2e    : proposals/s through the plug-in call with HOST (pinned) buffers: H2D of the start
         points + D2H of (u, v, logl, counters) inside the timed region, every step.
roofline: algorithmic bytes B_rwalk(n) = 16 n^2 + 24 n per proposal (SURVEY.md section 8d)
         x proposals per launch / kernel time (events on the launch stream) vs measured HBM peak.
cpu_baseline / --impl reference: the oracle port of the reference's pure-Python rwalk chain
         (oracle/samplers.py) on the host cores, bounded sample.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

# one BLAS / OpenMP thread per process BEFORE numpy loads: the CPU arm runs one process per core, and a 50 x 50
# mat-vec must not fan out into a thread team in each of them
for _v in ('OMP_NUM_THREADS', 'OPENBLAS_NUM_THREADS', 'MKL_NUM_THREADS'):
    os.environ.setdefault(_v, '1')
# the replicas of the ensemble block drive one stream each: give them hardware queues of their own (default 8)
os.environ.setdefault('CUDA_DEVICE_MAX_CONNECTIONS', '32')

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 56432
WORKLOADS = {
    # name: (ndim, nlive, sampler, steps-per-chain, bound)
    'c2': dict(ndim=50, nlive=2000, sample='rwalk', walks=70, bound='multi',
               desc="50-D correlated Gaussian, bound=multi, sample=rwalk, nlive=2000"),
}
METRIC = "rwalk proposals/sec (50-D correlated Gaussian, multi-ellipsoid bound)"


# ----------------------------------------------------------------------------- workload
def make_state(ndim, nlive, seed=SEED):
    """Synthetic mid-run nested-sampling state: `nlive` points uniform inside the iso-likelihood
    ellipsoid (v-mu)^T Cinv (v-mu) < r^2 with r^2 = ndim, so every live point has
    logl > loglstar = lnorm - r^2/2 (what the live set looks like when the run has
    compressed to the bulk of the posterior)."""
    rng = np.random.default_rng(seed)
    Cm = np.full((ndim, ndim), 0.4)
    np.fill_diagonal(Cm, 1.0)
    L = np.linalg.cholesky(Cm)
    z = rng.standard_normal((nlive, ndim))
    z *= (rng.random(nlive)**(1. / ndim) / np.linalg.norm(z, axis=1))[:, None]
    r = math.sqrt(ndim)
    v = r * z @ L.T
    u = (v + 5.0) / 10.0
    lnorm = -0.5 * (math.log(2 * math.pi) * ndim + np.linalg.slogdet(Cm)[1])
    loglstar = lnorm - 0.5 * r * r
    return np.ascontiguousarray(u), loglstar


def config_block(cfg, Q):
    """`config` of the JSON line -- the SAME dict in both arms (the driver compares them)."""
    return {"workload": cfg['desc'], "queue_chains_per_gpu": int(Q), "walks": int(cfg['walks']),
            "l2": "GPU arm: flushed (256 MB memset) between timed iterations"}


def algorithmic_bytes(n):
    return 16 * n * n + 24 * n      # SURVEY.md section 8(d): B_rwalk(n), GAUSS_PREC likelihood


def host_cores():
    """Cores this process may use: the scheduler affinity mask, capped by the cgroup CPU quota (a container
    lease can expose 128 CPUs in the mask and grant 8 of them in /sys/fs/cgroup/cpu.max)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    quota = None
    try:
        with open('/sys/fs/cgroup/cpu.max') as f:                       # cgroup v2
            q, per = f.read().split()
        if q != 'max':
            quota = float(q) / float(per)
    except Exception:
        try:                                                            # cgroup v1
            with open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us') as f:
                q = float(f.read())
            with open('/sys/fs/cgroup/cpu/cpu.cfs_period_us') as f:
                per = float(f.read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    if quota is not None:
        n = max(1, min(n, int(math.floor(quota + 0.5))))
    return n


def pick_process_count(cfg, pool_factory, cores, state, kind, seconds=1.5):
    """The process count that actually maximises the CPU arm's throughput on THIS box.  A quota is not the only
    way a lease is CPU-starved (round-1 BENCH: 128 CPUs visible, 7x one core delivered): time a short sample at
    cores, cores/2, cores/4, ... and keep the best, so the reference arm is never handicapped by
    oversubscription.  Returns (processes, {processes: proposals/s})."""
    tried = {}
    for p in sorted({cores, max(1, cores // 2), max(1, cores // 4), max(1, cores // 8)}, reverse=True):
        pool = pool_factory(p)
        try:
            tried[p] = cpu_sample(cfg, seconds, pool, p, state, kind)[0]
        finally:
            if pool is not None:
                pool.close()
    best = max(tried, key=tried.get)
    return best, tried


# ----------------------------------------------------------------------------- CPU arm
_REF = {}


def reference_kind():
    """"reference" when the unmodified dynesty is importable (a dynesty checkout or its git-ignored copy
    oracle/_ref, oracle/refshim.py), else "port" (the oracle)."""
    from oracle import refshim
    return 'reference' if refshim.available() else 'port'


def _cpu_worker_ref(args):
    """The UNMODIFIED reference: dynesty.internal_samplers.RWalkSampler.sample(SamplerArgument)
    per chain -- the static method dynesty's pool maps over the queue (sampler.py:717) -- with
    utils.LogLikelihood around the notebook's numpy likelihood and numpy's PCG64 generator."""
    os.environ.setdefault('OMP_NUM_THREADS', '1')
    u0s, loglstar, axes, scale, walks, chain0, ndim = args
    if 'mod' not in _REF:
        from oracle import refshim
        dynesty = refshim.import_reference()
        from dynesty import internal_samplers as RIS, utils as RU
        Cm = np.full((ndim, ndim), 0.4)
        np.fill_diagonal(Cm, 1.0)
        Cinv = np.linalg.inv(Cm)
        lnorm = -0.5 * (math.log(2 * math.pi) * ndim + np.linalg.slogdet(Cm)[1])
        _REF.update(mod=RIS, ptform=lambda u: 10. * u - 5.,
                    logl=RU.LogLikelihood(lambda x: -0.5 * np.dot(x, np.dot(Cinv, x)) + lnorm, ndim))
    RIS = _REF['mod']
    kw = {'walks': walks, 'ncdim': ndim, 'nonbounded': None, 'periodic': None, 'reflective': None}
    nacc = 0
    for i, u0 in enumerate(u0s):
        a = RIS.SamplerArgument(u=u0, loglstar=loglstar, axes=axes, scale=scale, prior_transform=_REF['ptform'],
                                loglikelihood=_REF['logl'], rseed=SEED + chain0 + i, kwargs=kw)
        r = RIS.RWalkSampler.sample(a)
        nacc += r.proposal_stats['n_accept']
    return len(u0s) * walks, nacc


def _cpu_worker(args):
    """Oracle port of the reference's per-chain pure-Python loop (what dynesty.pool.Pool maps)."""
    os.environ.setdefault('OMP_NUM_THREADS', '1')
    from oracle import samplers as OS, philox, likelihoods as OL
    u0s, loglstar, axes, scale, walks, chain0, ndim = args
    m = OL.gauss_corr(ndim, 0.4, 5.0)
    nacc = 0
    for i, u0 in enumerate(u0s):
        r = OS.rwalk_chain(u0, loglstar, axes, scale, m, philox.NumpyStream(SEED, chain0 + i), walks)
        nacc += r['n_accept']
    return len(u0s) * walks, nacc


def cpu_sample(cfg, target_seconds, pool, cores, state=None, kind='port'):
    """Times the reference's (kind="reference") or the oracle's (kind="port") rwalk chains on
    `cores` processes for ~target_seconds."""
    from oracle import bounding as OB
    worker = _cpu_worker_ref if kind == 'reference' else _cpu_worker
    u, loglstar = state if state is not None else make_state(cfg['ndim'], cfg['nlive'])
    ell = OB.bounding_ellipsoid(u)
    ell.scale_to_logvol(ell.logvol + math.log(1.25))
    rng = np.random.default_rng(1)
    scale, walks, n = 0.15, cfg['walks'], cfg['ndim']
    # pilot on every process at once (import + contention included) to size the bounded sample
    pilot = [(u[:4], loglstar, ell.axes, scale, walks, c * 4, n) for c in range(cores)]
    _ = pool.map(worker, pilot) if pool is not None else [worker(t) for t in pilot]    # imports, untimed
    t0 = time.perf_counter()
    _ = pool.map(worker, pilot) if pool is not None else [worker(t) for t in pilot]
    per_chain = (time.perf_counter() - t0) / 4
    per_core = max(4, min(int(target_seconds / per_chain), 20000))
    tasks = []
    for c in range(cores):
        starts = u[rng.integers(len(u), size=per_core)]
        tasks.append((starts, loglstar, ell.axes, scale, walks, 10**6 + c * per_core, n))
    t0 = time.perf_counter()
    res = pool.map(worker, tasks) if pool is not None else [worker(t) for t in tasks]
    dt = time.perf_counter() - t0
    nprop = sum(r[0] for r in res)
    return nprop / dt, nprop, dt, per_core * cores


def run_reference(args, cfg):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import multiprocessing as mp
    visible = host_cores()
    os.environ['OMP_NUM_THREADS'] = '1'
    state = make_state(cfg['ndim'], cfg['nlive'])
    kind = reference_kind()
    mk = lambda p: mp.get_context('fork').Pool(p) if p > 1 else None
    cores, tried = pick_process_count(cfg, mk, visible, state, kind)
    pool = mk(cores)
    per_step = float(os.environ.get('B2N_BENCH_CPU_SECONDS', max(1.0, min(20.0, 120.0 / max(1, args.steps + args.warmup)))))
    for _ in range(args.warmup):
        cpu_sample(cfg, per_step, pool, cores, state, kind)
    tot_p = tot_t = 0.0
    nchains = 0
    for _ in range(args.steps):
        _, p, t, nch = cpu_sample(cfg, per_step, pool, cores, state, kind)
        tot_p += p
        tot_t += t
        nchains = nch
    if pool is not None:
        pool.close()
    val = tot_p / tot_t
    who = ("dynesty RWalkSampler.sample (unmodified reference)" if kind == 'reference'
           else "oracle rwalk")
    sample = "%d %s chains x %d walks per step on %d processes" % (nchains, who, cfg['walks'], cores)
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "proposals/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_t / max(args.steps, 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": config_block(cfg, args.chains or cfg['nlive']),
            "run": {"chains_per_step": nchains, "processes": cores},
            "cpu_baseline": {"value": val, "unit": "proposals/s", "cores": cores, "kind": kind, "sample": sample,
                             "cores_visible": visible,
                             "process_count_scan": {str(k): round(v, 1) for k, v in sorted(tried.items())}},
            "e2e": {"value": val, "unit": "proposals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.p = None
        try:
            self.p = subprocess.Popen(['nvidia-smi', '-i', str(device), '--query-gpu=' + self.Q,
                                       '--format=csv,noheader,nounits', '-lms', '20'],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            pass

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        out = self.p.communicate()[0]
        sm, mx, reasons = [], None, set()
        for ln in out.strip().splitlines():
            f = [x.strip() for x in ln.split(',')]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx = float(f[2])
            except ValueError:
                continue
            for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[4:8]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        load = sorted(sm)[len(sm) // 2:] if sm else []          # upper half = samples under load
        return {"sm_mhz": (sorted(load)[len(load) // 2] if load else None), "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------- GPU arm
RWALK_OUTPUTS = ('u', 'v', 'logl', 'n_accept', 'n_reject', 'ncall')


def dump_outputs(outdir, ctx, d_out, Q, n, fused_world):
    """--dump-outputs: what the last timed step returned to its caller -- rank 0's queue of Q chains (end point u,
    its prior transform v and logl, and the chain counters) -- as DIR/<name>.npy in float64 (the counters exactly).
    With the fused exchange the step writes into the peer window, so the rows are read from there."""
    if fused_world:
        o = ctx.peer_gathered(fused_world * Q, n, RWALK_OUTPUTS[3:])
        o = {k: v[:Q] for k, v in o.items()}
    else:
        o = {k: d_out[k].cpu().numpy() for k in RWALK_OUTPUTS}
    os.makedirs(outdir, exist_ok=True)
    for k in RWALK_OUTPUTS:
        np.save(os.path.join(outdir, k + '.npy'), np.ascontiguousarray(o[k], dtype=np.float64))


def e2e_plugin(args, cfg, ctx, model, u_live, loglstar, scale, Q, walks):
    """The plug-in path a dynesty user drives, timed per queue fill on HOST data (every H2D / D2H inside):
      prepare_sampler : B200RWalkSampler.prepare_sampler(points=<list of Q rows>, axes=<Q axes handles>, seeds) +
                        map(sample) -- what Sampler._fill_queue hands the sampler and gets back (Q SamplerReturn)
      dynesty_fill_queue : the UNMODIFIED reference's own Sampler._fill_queue (sampler.py:676-717) with
                        bound=B200MultiEllipsoid, sample=B200RWalkSampler, pool=B200Pool, queue_size=Q -- Q x
                        propose_live (start row, get_random_axes, bound.contains) + prepare_sampler + map; only
                        when the reference is importable (oracle/refshim.py)."""
    import importlib
    from dynesty_b200 import _lib, samplers as S, bounding as B
    from dynesty_b200.pool import B200Pool
    n, steps = cfg['ndim'], args.steps
    ctx.set_pointer_mode(_lib.PTR_HOST)
    out = {"unit": "proposals/s", "queue_size": Q, "walks": walks}
    rng = np.random.default_rng(SEED)
    bound = B.B200MultiEllipsoid(n, ctx=ctx)
    bound.update(u_live, rstate=rng)
    bound.scale_to_logvol(bound.logvol + math.log(1.25))
    smp = S.B200RWalkSampler(model=model, ndim=n, ncdim=n, walks=walks, ctx=ctx)
    smp.scale = scale

    def inputs():       # what dynesty's _fill_queue builds before it calls the sampler (the CALLER's cost, not timed here)
        starts = rng.integers(len(u_live), size=Q)
        pts = [u_live[i] for i in starts]
        axes = [bound.get_random_axes(rng) for _ in range(Q)]
        seeds = np.random.SeedSequence(rng.integers(0, 2**63 - 1, size=4)).spawn(Q)
        return pts, axes, seeds

    def fill(pts, axes, seeds):
        a = smp.prepare_sampler(loglstar=loglstar, points=pts, axes=axes, seeds=seeds, nested_sampler=None)
        return list(map(smp.sample, a))
    for _ in range(3):
        fill(*inputs())
    dt = dt_in = 0.0
    for _ in range(steps):
        t0 = time.perf_counter()
        args_ = inputs()
        t1 = time.perf_counter()
        fill(*args_)
        dt += time.perf_counter() - t1
        dt_in += t1 - t0
    out["prepare_sampler"] = {"value": Q * walks * steps / dt, "ms_per_fill": 1e3 * dt / steps,
                              "caller_input_ms_per_fill": 1e3 * dt_in / steps,
                              "note": "prepare_sampler + map(sample) only; caller_input_ms = building Q start rows, Q axes handles "
                                      "and SeedSequence.spawn(Q) the way dynesty's _fill_queue does (29 ms of it is the spawn)"}
    from oracle import refshim
    if not refshim.available():
        out["dynesty_fill_queue"] = None
        return out
    dynesty = refshim.import_reference()
    import dynesty_b200._compat as c
    importlib.reload(c)                      # the mirrors must subclass dynesty's own Bound / InternalSampler
    importlib.reload(B)
    importlib.reload(S)
    v_live, l_live = model.evaluate(u_live, ctx=ctx)
    ns = dynesty.NestedSampler(model.loglikelihood, model.prior_transform, n, nlive=len(u_live),
                               bound=B.B200MultiEllipsoid(n, ctx=ctx),
                               sample=S.B200RWalkSampler(model=model, walks=walks, ctx=ctx), pool=B200Pool(Q), queue_size=Q,
                               live_points=[u_live, v_live, l_live], first_update={'min_ncall': 0, 'min_eff': 100.},
                               rstate=np.random.default_rng(SEED),
                               use_pool={'prior_transform': False, 'loglikelihood': False})
    ns.update_bound_if_needed(loglstar, force=True)      # first bound: built on the GPU through the Bound seam
    ns.internal_sampler.scale = scale
    mine = [0.0]
    orig = ns.internal_sampler.prepare_sampler

    def timed_prepare(**kw):                             # how much of a fill is spent inside the plug-in
        t = time.perf_counter()
        r = orig(**kw)
        mine[0] += time.perf_counter() - t
        return r
    ns.internal_sampler.prepare_sampler = timed_prepare
    for _ in range(3):
        ns.nqueue = 0
        ns._fill_queue(loglstar)
    mine[0] = 0.0
    t0 = time.perf_counter()
    for _ in range(steps):
        ns.nqueue = 0
        ns._fill_queue(loglstar)
    dt = time.perf_counter() - t0
    assert len(ns.queue) == Q and all(r.logl > loglstar for r in ns.queue[:50])
    out["dynesty_fill_queue"] = {"value": Q * walks * steps / dt, "ms_per_fill": 1e3 * dt / steps,
                                 "ms_per_fill_inside_the_plugin": 1e3 * mine[0] / steps,
                                 "ms_per_fill_dynesty_python": 1e3 * (dt - mine[0]) / steps,
                                 "sampler": "unmodified dynesty.NestedSampler with the B200 bound / sampler / pool",
                                 "note": "dynesty's own per-slot Python (rstate.choice, get_random_axes, contains, SeedSequence.spawn) "
                                         "is the part outside the plug-in; it is why dynesty_b200.nested proposes a whole queue at once"}
    return out


def run_b200(args, cfg):
    import torch
    import torch.distributed as dist
    from dynesty_b200 import _lib, ops, likelihoods as DL, bounding as B

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus %d but WORLD_SIZE=%d" % (args.gpus, world))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    # stdout carries exactly ONE line (the JSON): while the benchmark runs, file descriptor 1 points at stderr,
    # so that banners printed by native libraries (NCCL's "NCCL version ..." goes to stdout) cannot precede it
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    ctx = _lib.Context(local)
    n, nlive, walks = cfg['ndim'], cfg['nlive'], cfg['walks']
    Q = args.chains or nlive
    model = DL.gauss_corr(n, 0.4, 5.0)
    mid = model.model_id(ctx)
    u_live, loglstar = make_state(n, nlive)

    # ---- the bounding half of the path: build + enlarge the bound on the GPU (timed separately)
    bound = B.B200MultiEllipsoid(n, ctx=ctx)
    t0 = time.perf_counter()
    bound.update(u_live, rstate=np.random.default_rng(SEED))
    bound.scale_to_logvol(bound.logvol + math.log(1.25))
    bound_ms_first = 1e3 * (time.perf_counter() - t0)
    t0 = time.perf_counter()
    for _ in range(3):
        bound.update(u_live, rstate=np.random.default_rng(SEED))
        bound.scale_to_logvol(bound.logvol + math.log(1.25))
    bound_ms = 1e3 * (time.perf_counter() - t0) / 3
    bound.make_resident()
    rng = np.random.default_rng(SEED + rank)

    # ---- buffers
    pin = lambda *s, dt=torch.float64: torch.empty(*s, dtype=dt).pin_memory()
    h_u0 = pin(Q, n)
    h_live = pin(nlive, n)                      # the live set, pinned: the kernels read their start rows from it in place
    h_live.numpy()[:] = u_live
    h_out = dict(u=pin(Q, n), v=pin(Q, n), logl=pin(Q), n_accept=pin(Q, dt=torch.int32),
                 n_reject=pin(Q, dt=torch.int32), ncall=pin(Q, dt=torch.int32))
    h_np = {k: t.numpy() for k, t in h_out.items()}
    d_live = torch.from_numpy(u_live).to(dev)
    d_u0 = torch.empty(Q, n, dtype=torch.float64, device=dev)
    d_pack = torch.empty(Q * n + Q, dtype=torch.float64, device=dev)     # (u | logl): ONE all-gather per fill
    d_out = dict(u=d_pack[:Q * n].view(Q, n), v=torch.empty(Q, n, dtype=torch.float64, device=dev),
                 logl=d_pack[Q * n:],
                 n_accept=torch.empty(Q, dtype=torch.int32, device=dev),
                 n_reject=torch.empty(Q, dtype=torch.int32, device=dev),
                 ncall=torch.empty(Q, dtype=torch.int32, device=dev))
    fused = world > 1 and args.exchange == 'fused'
    if world > 1:
        g_pack = torch.empty(world * (Q * n + Q), dtype=torch.float64, device=dev)
    if fused:
        # the exchange step fused into the kernel: finished chains are stored into every rank's
        # window over NVLink and the kernel ends with a cross-GPU arrive/wait (csrc/b2n_peer.cu)
        from dynesty_b200.dist import Comm
        Comm(dev).attach_peer(ctx, world * Q, n)
        hg_out = dict(u=pin(world * Q, n), v=pin(world * Q, n), logl=pin(world * Q),
                      n_accept=pin(world * Q, dt=torch.int32), n_reject=pin(world * Q, dt=torch.int32),
                      ncall=pin(world * Q, dt=torch.int32))
        hg_np = {k: t.numpy() for k, t in hg_out.items()}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)       # > 126 MB L2
    # one explicit (non-default) stream shared by torch and the library, so that torch's CUDA
    # events bracket the library's launches (a NULL handle would mean "library-owned stream")
    stream = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    ctx.set_stream(stream.cuda_stream)
    ctx.set_timing(True)

    state = dict(scale=0.2, chain=0)

    def propose():
        starts = rng.integers(nlive, size=Q)
        ell = bound.random_ells(rng, Q)
        return starts, ell

    def step_host():
        """The plug-in call with host buffers (what Sampler._fill_queue does per fill): the start rows are named by
        index and read by the kernel from the (pinned) live set in place -- b2n_set_start_rows -- instead of being
        gathered into a block by the caller first (np.take: 40 us of a 0.32 ms step); --gather-starts restores that."""
        starts, ell = propose()
        if args.gather_starts:
            np.take(u_live, starts, axis=0, out=h_u0.numpy(), mode='clip')    # ('raise' buffers `out`: 3x slower)
            src, kw = h_u0.numpy(), {}
        else:
            src, kw = h_live.numpy(), dict(start_rows=starts.astype(np.int32, copy=False))
        ctx.set_pointer_mode(_lib.PTR_HOST)
        c0 = state['chain']
        state['chain'] += Q * world
        if fused:
            # every rank's WINDOW (HBM) receives the whole queue inside the kernel; only rank 0 -- the owner of the
            # nested-sampling bookkeeping -- copies it to its host, the other ranks' hosts receive nothing
            o = ops.rwalk_batch(mid, src, loglstar, state['scale'], walks, SEED, chain0=c0 + rank * Q,
                                ell=ell, ctx=ctx, out=hg_np if rank == 0 else ops.NO_OUT, peer=(rank * Q, world * Q), **kw)
            if rank != 0:
                return None
            return {k: v[rank * Q:(rank + 1) * Q] for k, v in o.items()}
        o = ops.rwalk_batch(mid, src, loglstar, state['scale'], walks, SEED, chain0=c0 + rank * Q,
                            ell=ell, ctx=ctx, out=h_np, **kw)
        return o

    def prep_dev():
        """Inputs of the next device-resident step: start points gathered from the live set in HBM
        (outside the timed events: `value` starts with its inputs resident)."""
        starts, ell = propose()
        torch.index_select(d_live, 0, torch.from_numpy(starts).to(dev, non_blocking=True), out=d_u0)
        return ell

    def step_dev(ell=None):
        """Same step with the inputs already resident in HBM (device pointers, async)."""
        if ell is None:
            ell = prep_dev()
        ctx.set_pointer_mode(_lib.PTR_DEVICE)
        c0 = state['chain']
        state['chain'] += Q * world
        if fused:           # the exchange step of the sharded path, inside the kernel
            ops.rwalk_batch(mid, d_u0, loglstar, state['scale'], walks, SEED, chain0=c0 + rank * Q, ell=ell,
                            ctx=ctx, out=ops.NO_OUT, peer=(rank * Q, world * Q))
            return
        ops.rwalk_batch(mid, d_u0, loglstar, state['scale'], walks, SEED, chain0=c0 + rank * Q, ell=ell,
                        ctx=ctx, out=d_out)
        if world > 1:       # --exchange nccl: one packed all-gather of (u | logl) after the kernel
            dist.all_gather_into_tensor(g_pack, d_pack)

    # ---- warm-up: also tunes the proposal scale with the reference's rule (internal_samplers.py:491)
    clocks = ClockSampler(local)         # samples every 20 ms from here to the end of the timed regions
    def sync_scale(acc_frac):
        """rank 0 tunes the proposal scale (it alone sees the counters on its host); every rank uses its value"""
        t = torch.tensor([acc_frac if acc_frac is not None else 0.0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.broadcast(t, 0)
        return float(t[0])

    for _ in range(max(args.warmup, 3)):
        o = step_host()
        fr = None if o is None else float(o['n_accept'].sum() / (o['n_accept'].sum() + o['n_reject'].sum()))
        fr = sync_scale(fr)
        state['scale'] *= math.exp((fr - 0.5) / n / 0.5)
    for _ in range(3):
        o = step_host()
    accept_frac = sync_scale(None if o is None else float(o['n_accept'].sum() / (o['n_accept'].sum() + o['n_reject'].sum())))
    # ---- N > 1: the gathered rows must BE what a single GPU computes for the same chain ids (rank 0 recomputes
    #      the rows of the last rank locally and compares them with what arrived in its window)
    gather_check = None
    if fused:
        starts_c, ell_c = propose()
        np.take(u_live, starts_c, axis=0, out=h_u0.numpy(), mode='clip')
        allq = [None] * world
        dist.all_gather_object(allq, (h_u0.numpy().copy(), ell_c))
        ctx.set_pointer_mode(_lib.PTR_HOST)
        c0 = state['chain']
        state['chain'] += Q * world
        o = ops.rwalk_batch(mid, h_u0.numpy(), loglstar, state['scale'], walks, SEED, chain0=c0 + rank * Q, ell=ell_c,
                            ctx=ctx, out=hg_np if rank == 0 else ops.NO_OUT, peer=(rank * Q, world * Q))
        if rank == 0:
            r = world - 1
            got = {k: v[r * Q:(r + 1) * Q].copy() for k, v in o.items()}
            loc = ops.rwalk_batch(mid, allq[r][0], loglstar, state['scale'], walks, SEED, chain0=c0 + r * Q, ell=allq[r][1],
                                  ctx=ctx)
            same = all(np.array_equal(got[k], loc[k]) for k in ('u', 'v', 'logl', 'n_accept', 'n_reject', 'ncall'))
            gather_check = {"rows_of_rank": r, "bit_identical_to_local_recompute": bool(same)}
            if not same:
                raise SystemExit("gathered rows differ from a local recomputation")
        dist.barrier()
    # clock ramp: ~0.7 s of the same kernel before timing, so that the nvidia-smi sampler has
    # samples under load.  N>1: a FIXED step count (every rank must issue the same exchanges).
    # The timed steps start from the proposal RNG and chain counter as they are here, so that
    # their inputs do not depend on how many ramp steps fit into the time.
    rng_state, chain_next = rng.bit_generator.state, state['chain']
    if world > 1:
        for _ in range(2500):
            step_dev()
    else:
        t_ramp = time.perf_counter() + args.ramp
        while time.perf_counter() < t_ramp:
            step_dev()
    torch.cuda.synchronize()
    rng.bit_generator.state, state['chain'] = rng_state, chain_next

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- timed: device-resident (value + roofline)
    launches0 = ctx.launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    kern_ms = []
    barrier()
    for a, b in ev:
        ell = prep_dev()
        flush.zero_()                        # L2 flush between timed iterations (outside the events)
        a.record(stream)
        step_dev(ell)
        b.record(stream)
        b.synchronize()
        kern_ms.append(ctx.last_kernel_ms())
    barrier()
    dev_ms = sum(a.elapsed_time(b) for a, b in ev)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ctx, d_out, Q, n, world if fused else 0)
    # ---- timed: end to end through the plug-in call with host buffers
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_host()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    barrier()
    launches = ctx.launch_count() - launches0
    clk = clocks.stop()
    if fused:
        ctx.peer_check()                     # raises if any in-kernel exchange ever timed out

    # ---- e2e through the reference-facing PLUG-IN objects: what dynesty's Sampler._fill_queue costs per fill
    plugin = None
    if rank == 0:
        try:
            plugin = e2e_plugin(args, cfg, ctx, model, u_live, loglstar, state['scale'], Q, walks)
        except Exception as e:                       # never lose the contract line over the extra measurement
            plugin = {"error": repr(e)[:200]}
    if world > 1:
        dist.barrier()
    # ---- measured FP64 ceilings of this GPU (the kernel's real bound; nothing quoted)
    ctx.set_pointer_mode(_lib.PTR_HOST)
    fp64 = None
    if rank == 0:
        fma_tf, fma_ms = ops.fp64_peak('fma', 20000, ctx=ctx)
        mma_tf, mma_ms = ops.fp64_peak('mma', 20000, ctx=ctx)
        fp64 = {"fma_tflops": fma_tf, "mma_tflops": mma_tf, "fma_ms": fma_ms, "mma_ms": mma_ms}

    t = torch.tensor([dev_ms, e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_s = float(t[0]), float(t[1])
    props_per_step = Q * walks * world
    value = props_per_step * args.steps / (dev_ms * 1e-3)
    e2e = props_per_step * args.steps / e2e_s

    line = None
    if rank == 0:
        peaks, peak_src = None, "fallback 6650 GB/s (B200_PROFILING.md)"
        try:
            with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
                peaks = json.load(f)
            peak, peak_src = float(peaks['hbm_gbs']), "MEASURED_PEAKS.json hbm_gbs (burst copy)"
        except Exception:
            peak = 6650.0
        kms = float(np.mean(kern_ms))
        achieved = algorithmic_bytes(n) * Q * walks / (kms * 1e-3) / 1e9
        # which lock-step kernel the library runs for this shape (csrc/b2n_rwalk.cu: B2N_RWALK_WARPS, default 12)
        ws = os.environ.get('B2N_RWALK_WARPS', '12') == '12'
        kernel_key = 'rwalk_mmaws_kernel' if ws else 'rwalk_mma_kernel'
        kernel_name = ("rwalk_mmaws_kernel<KT=13, setmaxnreg 88/64, plain>: 8 step + 4 draw warps per 8 chains, ring 2 x 8" if ws
                       else "rwalk_mma_kernel<GAUSS_PREC, KT=13, 8 chains/CTA, ring 8>")
        traffic = None          # DRAM bytes per launch of this kernel from the committed ncu --set full capture
        try:                    # (profiles/traffic.json: a constant of the capture, NOT measured in this run)
            with open(os.path.join(ROOT, 'profiles', 'traffic.json')) as f:
                traffic = json.load(f)[kernel_key]['dram_bytes_per_launch'] if Q == 2000 else None
        except Exception:
            pass
        flops_pp = 4 * n * n + 7 * n                      # SURVEY 8(d): flop per proposal
        mma_flops_pp, fma_flops_pp = 4 * n * n, 7 * n     # the two contractions (DMMA) / everything else (DFMA)
        ach_tf = flops_pp * Q * walks / (kms * 1e-3) / 1e12
        # time the launch would take if both pipes ran at their measured ceilings back to back
        t_floor_ms = 1e3 * Q * walks * (mma_flops_pp / (fp64["mma_tflops"] * 1e12) + fma_flops_pp / (fp64["fma_tflops"] * 1e12))
        line = {
            "metric": METRIC, "value": value, "unit": "proposals/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_block(cfg, Q),
            "run": {"nells": int(bound.nells), "accept_fraction": round(accept_frac, 3), "scale": round(state['scale'], 4),
                    "exchange": ("fused into the kernel: NVLink peer stores + in-kernel arrive/wait" if fused else
                                 ("NCCL all-gather after the kernel" if world > 1 else "none (1 GPU)")),
                    "bound_update_ms": round(bound_ms, 3), "bound_update_first_ms": round(bound_ms_first, 2)},
            "e2e": {"value": e2e, "unit": "proposals/s",
                    "h2d_bytes_per_step": Q * n * 8 + Q * 4 + 16 * (Q // 8 + 1) + (0 if args.gather_starts else Q * 4),
                    "start_points": ("gathered by the caller into a pinned block (np.take)" if args.gather_starts else
                                     "by index: the kernel reads rows idx[q] of the pinned live set in place (b2n_set_start_rows)"),
                    "d2h_bytes_per_step": (world if fused else 1) * (2 * Q * n * 8 + Q * 8 + 3 * Q * 4),
                    "bytes_are": ("rank 0 (the owner of the sampler state receives the whole queue; the other ranks' hosts "
                                  "receive nothing)" if fused else "per rank")},
            "gpu_launches": int(launches),
            "accepted_proposals_per_s": value * accept_frac,      # SURVEY 8(d): rwalk n_accept / wall
            # The dominant kernel's two mat-vecs per proposal are FP64 tensor-core MMAs (mma.m8n8k4.f64) on
            # register-resident matrices: its bound is the FP64 pipes, not HBM.  Both ceilings are MEASURED in
            # this run by the library's own microbenchmark (b2n_fp64_peak: 16 independent chains per thread on
            # every SM); `peak` is the measured FP64 MMA rate, which carries 97 % of the flops.
            "roofline": {"bound": "tensor", "achieved": ach_tf, "peak": fp64["mma_tflops"], "unit": "TFLOP/s",
                         "frac": ach_tf / fp64["mma_tflops"], "traffic": traffic, "traffic_unit": "bytes/launch",
                         "traffic_source": "profiles/traffic.json (ncu --set full capture of this kernel at this size; a "
                                           "constant, not measured in this run)",
                         "kernel": kernel_name, "kernel_ms": kms,
                         "flops_per_proposal": flops_pp, "flops_per_launch": flops_pp * Q * walks,
                         "peak_source": "measured in this run: FP64 mma.m8n8k4 rate of this GPU (b2n_fp64_peak kind 1)",
                         "fp64_fma_peak_tflops": fp64["fma_tflops"], "fp64_mma_peak_tflops": fp64["mma_tflops"],
                         "pipes_floor_ms": t_floor_ms, "frac_of_pipes_floor": t_floor_ms / kms,
                         "note": ("MEASURED_PEAKS.json holds HBM and bf16 numbers only; this kernel computes in FP64, so the "
                                  "FP64 ceilings are measured here.  pipes_floor_ms = launch time with both FP64 pipes at their "
                                  "measured ceilings; the rest is the FP64 of the draws (Philox + Box-Muller) and the serial chain "
                                  "phases of a step, DESIGN.md 9.6")},
            # SURVEY 8(d)'s no-reuse byte model (both 20 KB matrices charged to every proposal) against the measured
            # HBM copy peak.  > 1 by construction for a kernel that keeps the matrices in registers: kept as the
            # figure the survey defines, not as evidence.
            "roofline_hbm_model": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                                   "algorithmic_bytes_per_proposal": algorithmic_bytes(n),
                                   "algorithmic_bytes_per_launch": algorithmic_bytes(n) * Q * walks, "peak_source": peak_src},
            "e2e_plugin": plugin,
            "gather_check": gather_check,
            "clocks": clk,
        }
    if world > 1:
        dist.barrier()

    # ---- the second half of the metric, and throughput AT THE SAME OPERATING POINT: an ensemble of full C2 runs
    #      (one per seed) with the rounds on the device at the batch that reproduces the reference's logZ
    #      (nlive/40), the replicas running concurrently on every GPU (dynesty_b200/replicas.py).  The ensemble is
    #      FIXED (args.ensemble runs) whatever --gpus is: its calls/s over N = 1, 2, 4, 8 is the strong-scaling curve.
    if args.ensemble:
        from dynesty_b200 import replicas
        ctx.set_timing(False)
        ctx.set_pointer_mode(_lib.PTR_HOST)
        comm = None
        if world > 1:
            from dynesty_b200.dist import Comm
            comm = Comm(dev)
        batch = args.logz_batch or max(1, nlive // 40)
        seeds = list(range(SEED, SEED + args.ensemble))
        rkw = dict(nlive=nlive, bound=cfg['bound'], sample=cfg['sample'], sampler_kwargs=dict(walks=walks), device=local,
                   max_in_flight=args.in_flight, chain_pack=args.chain_pack, comm=comm, batch=batch, errors='record')
        # the contexts (stream, scratch, device run state) are a pool that outlives the ensemble, as in a service that
        # keeps its GPUs: created and warmed up -- one run per context -- outside the timed region
        mine = len(seeds[rank::world])
        pool = replicas.ContextPool(local, max(1, min(args.in_flight, mine)), args.chain_pack)
        rkw['pool'] = pool
        replicas.run_replicas(model, seeds[:min(len(seeds), args.in_flight * world)], **rkw)
        barrier()
        t0 = time.perf_counter()
        outs, _ = replicas.run_replicas(model, seeds, **rkw)
        barrier()
        tens = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        pool.close()
        del rkw['pool']
        if world > 1:
            dist.all_reduce(tens, op=dist.ReduceOp.MAX)
        ens_wall = float(tens[0])
        if rank == 0:
            summ = replicas.summarize(outs, ens_wall)
            failed = [o for o in outs if 'error' in o]
            outs = [o for o in outs if 'error' not in o]
            runs = [{k: (round(v, 4) if isinstance(v, float) else v) for k, v in o.items()} for o in outs]
            line["full_runs"] = {
                "what": ("%d full C2 nested-sampling runs (seeds %d..%d), device rounds (b2n_ns_run) with batch = %d, %d "
                         "replicas in flight per GPU; proposals/s and logZ come from THE SAME runs" %
                         (len(seeds), seeds[0], seeds[-1], batch, args.in_flight)),
                "scaling": "strong (the ensemble is fixed; ranks take seeds[rank::world])",
                "batch": batch, "replicas": len(seeds), "failed_replicas": [f["error"] for f in failed][:4], "in_flight_per_gpu": args.in_flight, "chains_per_cta": args.chain_pack,
                "n_gpus": world,
                "wall_s": ens_wall, "proposals_per_s": summ["calls_per_s"], "calls_per_s": summ["calls_per_s"],
                "iterations_per_s": summ["niter"] / ens_wall, "run_wall_s_mean": summ["run_wall_s_mean"],
                "logz_mean": summ["logz_mean"], "logz_std": summ["logz_std"], "truth": model.logz_truth,
                "abs_err_mean": abs(summ["logz_mean"] - model.logz_truth),
                "runs": runs[:8], "logz_all": [round(o["logz"], 4) for o in outs]}
            try:        # the UNMODIFIED reference on this config (CPU, serial), recorded by scripts/ref_c2_run.py
                with open(os.path.join(ROOT, 'profiles', 'ref_c2_rwalk_nlive2000.jsonl')) as f:
                    ref = [json.loads(x) for x in f if x.strip()]
                rz = np.array([r["logz"] for r in ref])
                line["full_runs"]["reference"] = {
                    "logz_mean": float(rz.mean()), "logz_std": float(rz.std(ddof=1)), "runs": len(rz),
                    "wall_s_mean": float(np.mean([r["wall"] for r in ref])),
                    "calls_per_s_one_core": float(np.mean([r["ncall"] / r["wall"] for r in ref])),
                    "source": "profiles/ref_c2_rwalk_nlive2000.jsonl (dynesty, 1 CPU core, build container)"}
                line["full_runs"]["mean_minus_reference_mean"] = float(summ["logz_mean"] - rz.mean())
            except Exception:
                pass
        if world == 1 and args.solo:          # latency of ONE run with nothing else on the GPU
            o1, w1 = replicas.run_replicas(model, [SEED], **dict(rkw, max_in_flight=1, chain_pack=1))
            line["full_runs"]["solo_run"] = {"wall_s": w1, "calls_per_s": o1[0]["ncall"] / w1, "logz": o1[0]["logz"],
                                             "rounds_s": o1[0]["rounds_s"], "bound_s": o1[0]["bound_s"],
                                             "nbound": o1[0]["nbound"], "rounds": o1[0]["rounds"]}
    # ---- CPU baseline on the host cores (rank 0, N=1 only), bounded sample
    if rank == 0 and world == 1 and args.cpu_baseline:
        import multiprocessing as mp
        visible = host_cores()
        os.environ['OMP_NUM_THREADS'] = '1'
        kind = reference_kind()
        mk = lambda p: mp.get_context('fork').Pool(p) if p > 1 else None
        cores, tried = pick_process_count(cfg, mk, visible, (u_live, loglstar), kind, seconds=1.0)
        pool = mk(cores)
        v, p, tsec, nch = cpu_sample(cfg, 10.0, pool, cores, (u_live, loglstar), kind)
        if pool is not None:
            pool.close()
        v1, _, t1, nch1 = cpu_sample(cfg, 3.0, None, 1, (u_live, loglstar), kind)   # SURVEY 8(d): (i) one core, serial
        who = "dynesty RWalkSampler.sample (unmodified reference)" if kind == 'reference' else "oracle rwalk"
        line["cpu_baseline"] = {"value": v, "unit": "proposals/s", "cores": cores, "kind": kind,
                                "sample": "%d %s chains x %d walks (%.1f s) on %d processes" % (nch, who, walks, tsec, cores),
                                "one_core_value": v1, "one_core_sample": "%d chains (%.1f s), serial" % (nch1, t1),
                                "cores_visible": visible, "effective_cores": v / v1,
                                "process_count_scan": {str(k): round(x, 1) for k, x in sorted(tried.items())}}
    sys.stdout.flush()
    os.dup2(real_stdout, 1)
    os.close(real_stdout)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        os.dup2(2, 1)               # (teardown messages of native libraries: not on stdout either)
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='c2', choices=sorted(WORKLOADS))
    ap.add_argument('--chains', type=int, default=0, help='chains per step per GPU (default nlive)')
    ap.add_argument('--ensemble', type=int, default=512, help='full C2 runs (seeds) of the logZ / same-operating-point block; 0 = none')
    ap.add_argument('--in-flight', type=int, default=32, help='replicas in flight per GPU')
    ap.add_argument('--chain-pack', type=int, default=4, help='chains per CTA of the replicas (b2n_set_chain_pack)')
    ap.add_argument('--solo', type=int, default=1, help='N=1: also time one run alone on the GPU')
    ap.add_argument('--logz-batch', type=int, default=0, help='points replaced per device round (default nlive/40)')
    ap.add_argument('--cpu-baseline', type=int, default=1)
    ap.add_argument('--gather-starts', type=int, default=0, help='e2e: 1 = the caller gathers the start rows (np.take) instead of passing indices')
    ap.add_argument('--ramp', type=float, default=0.7, help='seconds of untimed steps before timing (clock ramp; 0 under ncu)')
    ap.add_argument('--exchange', default='fused', choices=['fused', 'nccl'],
                    help='N>1: how the finished chains reach every rank')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the outputs of the last timed device step as DIR/<name>.npy (float64)')
    args = ap.parse_args()
    cfg = WORKLOADS[args.workload]
    if args.impl == 'reference':
        run_reference(args, cfg)
    else:
        run_b200(args, cfg)


if __name__ == '__main__':
    main()
