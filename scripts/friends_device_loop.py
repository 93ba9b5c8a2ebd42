"""GPU: RadFriends / SupFriends bounds, one whole run per configuration with the rounds on the device
(run_nested(loop='device')) against the host loop (loop='host'): wall time, logZ +- err, ncall.  The SURVEY row is 2-D
shells, nlive 500, sample='unif', bound='balls' / 'cubes'; plus the 3-D Gaussian.  One JSON line per run, printed and
appended to <outdir>/friends_device_loop.jsonl; the first line records the GPU and its power limit.
usage: python scripts/friends_device_loop.py outdir"""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from dynesty_b200 import likelihoods as DL, nested  # noqa: E402


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clk = [x.strip() for x in q.split(',')]
    return dict(gpu=name, power_limit=power, max_sm_clock=clk)


def run(out, tag, model, loop, seed=56432, **kw):
    t0 = time.perf_counter()
    s = nested.NestedSampler(model, seed=seed, **kw)
    r = s.run_nested(loop=loop, dlogz=0.5)
    wall = time.perf_counter() - t0
    rec = dict(config=tag, loop=loop, bound=kw['bound'], sample=kw['sample'], nlive=kw['nlive'], seed=seed,
               wall_s=round(wall, 3), logz=round(float(r.logz[-1]), 4), logzerr=round(float(r.logzerr[-1]), 4),
               truth=model.logz_truth, ncall=int(r.ncall), niter=int(r.niter), nbound=int(r.nbound),
               batch=getattr(s, 'batch', None), rounds=getattr(s, 'device_rounds', None))
    if loop == 'device':
        rec.update(rounds_s=round(s.device_timing['rounds_s'], 3), bound_s=round(s.device_timing['bound_s'], 3))
    print(json.dumps(rec), flush=True)
    out.write(json.dumps(rec) + '\n')
    out.flush()


def main():
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    outdir = sys.argv[1]
    os.makedirs(outdir, exist_ok=True)
    with open(os.path.join(outdir, 'friends_device_loop.jsonl'), 'a') as out:
        info = gpu_info()
        print(json.dumps(info), flush=True)
        out.write(json.dumps(info) + '\n')
        # warm-up: library load, first launches, the first friends update (not recorded)
        nested.NestedSampler(DL.gauss_test3d(), nlive=100, bound='balls', sample='unif', seed=1).run_nested(
            loop='device', dlogz=5.0)
        for bound in ('balls', 'cubes'):
            for loop in ('device', 'host'):
                run(out, '2-D shells %s/unif nlive=500' % bound, DL.shells(2), loop, nlive=500, bound=bound,
                    sample='unif')
        for bound, sample in (('balls', 'unif'), ('cubes', 'rwalk')):
            for loop in ('device', 'host'):
                run(out, '3-D gauss %s/%s nlive=500' % (bound, sample), DL.gauss_test3d(), loop, nlive=500,
                    bound=bound, sample=sample)


if __name__ == '__main__':
    main()
