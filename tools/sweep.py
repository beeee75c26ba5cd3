#!/usr/bin/env python
"""Device-timed sweep of the step kernel over (env, envs, chained, streams, ...) in ONE process (bench.py's
Ring / measure, no e2e, no CPU baseline): one JSON line per case.  Tuning tool; bench.py is the record.

    python tools/sweep.py PointTSP-v0:65536:c1:s1 PointTTSP-v0:262144:c0:s2 ... [--steps 20000] [--warmup 50]
    case = env:envs[:cX][:sY][:pZ][:bK][:wW][:rR]   c = chained (0/1, default auto), s = streams, p = prefetch_every, b = layout bank size,
           w = sampler warps per SM, r = minimum number of ring replicas
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('cases', nargs='+')
    ap.add_argument('--steps', type=int, default=20000, help='timed steps per case')
    ap.add_argument('--warmup', type=int, default=50)
    ap.add_argument('--cfg', action='append', default=[])
    ap.add_argument('--no-auto-reset', action='store_true')
    a = ap.parse_args()
    import torch
    import combinatorial_rl_tasks_b200 as crl
    from combinatorial_rl_tasks_b200 import _lib
    dev = torch.device('cuda:0')
    torch.cuda.set_device(dev)
    peak, _ = bench.measured_peaks()
    for case in a.cases:
        parts = case.split(':')
        env_id, B = parts[0], int(parts[1])
        opt = {p[0]: int(p[1:]) for p in parts[2:]}
        args = argparse.Namespace(bank=opt.get('b', 0), prefetch_every=opt.get('p', 32), prefetch_warps=opt.get('w', 0),
                                  cfg=a.cfg, no_auto_reset=a.no_auto_reset, env=env_id, min_replicas=opt.get('r', 0))
        ring = bench.Ring(crl, _lib, args, env_id, B, dev, 0, chained=(None if 'c' not in opt else bool(opt['c'])),
                          streams=opt.get('s', 0))
        m = bench.measure(ring, a.steps, a.warmup, 1, None)
        d = bench.device_line(ring, m, 1, peak)
        c = ring.counters().cpu().numpy()
        print(json.dumps({'case': case, 'lib': os.environ.get('CRL_B200_LIB', 'default'), 'frac': round(d['frac'], 4),
                          'best': round(d['best_frac'], 4), 'mean': round(d['mean_frac'], 4), 'us_per_step': round(1e3 * d['ms_per_step'], 3),
                          'value': d['value'], 'chained': ring.chained, 'streams': ring.S, 'R': ring.R,
                          'episodes': c[1], 'resets_prefetched': c[4], 'resets_inline': c[5], 'chain_timeouts': c[7],
                          'timed_steps': m['timed_steps'], 'sampler_launches': ring.prefetch_launches}), flush=True)
        del ring
        torch.cuda.empty_cache()


if __name__ == '__main__':
    main()
