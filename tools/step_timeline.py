"""Per-step timeline of the graph-launched fused step: where the density branch ends against the gamete
branch.

Advances the bench.py workload `--presteps` steps, then records `--steps` graph-launched steps under
torch.profiler (CUDA activities) and writes, for every kernel of those steps, its stream, start and end
(µs, relative to the step's first kernel).  For every step it reports
  * pre_fork_us:     first kernel start -> end of k_density_counts (the fork);
  * density_us:      fork -> end of the density branch (k_ct_* and k_raster_* kernels);
  * gametes_us:      fork -> end of the last other kernel before k_death (k_gametes ... k_after_births);
  * exposed_us:      density_us - gametes_us (> 0: k_death waits for the density branch);
  * death_us:        k_death;
  * step_us:         first kernel start -> next step's first kernel start;
  * gaps:            idle stretches of a stream between two of its kernels longer than GAP_US, each with the
                     memset and memcpy nodes of the step that run inside it (the graph's non-kernel work).
`gap_median_us` gives the median of every such gap over the traced steps, keyed 'kernel -> kernel'.
The raster kernels have no row in bench.py's algorithmic-bytes table, so their bytes per launch (landscape
cells x bytes per cell) are reported here.  The library is the in-tree build, or GNX_B200_LIB.

  python tools/step_timeline.py --workload c2 --presteps 600 --steps 20 --out timeline_c2.json
"""
import argparse
import json
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

GAP_US = 2.0
# algorithmic bytes per landscape cell of the raster passes
RASTER_BYTES_PER_CELL = {'k_raster_N': 8, 'k_raster_d': 24, 'k_raster_Nd': 24}


def short_name(name):
    name = name.split('(')[0]
    name = name.split('<')[0]
    return name.replace('void ', '').strip()


def is_density(name):
    return name.startswith(('k_ct_', 'k_raster_'))


def split_steps(kernels):
    """kernels sorted by start -> one list per step (a step starts at k_move_key)."""
    steps, cur = [], None
    for k in kernels:
        if k['name'] == 'k_move_key':
            cur = []
            steps.append(cur)
        if cur is not None:
            cur.append(k)
    return steps


def step_gaps(ks, others):
    """Idle stretches of each stream between consecutive kernels, and the memset / memcpy nodes inside them."""
    out = []
    streams = sorted({k['stream'] for k in ks}, key=str)
    for st in streams:
        sk = [k for k in ks if k['stream'] == st]
        for a, b in zip(sk, sk[1:]):
            if b['start'] - a['end'] <= GAP_US:
                continue
            inside = [{'name': o['name'], 'kind': o['kind'], 'stream': o['stream'], 'us': o['end'] - o['start']}
                      for o in others if o['end'] > a['end'] and o['start'] < b['start']]
            out.append({'after': a['name'], 'before': b['name'], 'stream': st, 'us': b['start'] - a['end'],
                        'activity': inside})
    return out


def step_summary(ks, next_start):
    t0 = ks[0]['start']
    fork = next((k['end'] for k in ks if k['name'] == 'k_density_counts'), None)
    death = next((k for k in ks if k['name'] == 'k_death'), None)
    if fork is None or death is None:
        return None
    dens = [k for k in ks if is_density(k['name'])]
    gam = [k for k in ks if k['start'] >= fork and not is_density(k['name']) and k['name'] != 'k_death'
           and k['end'] <= death['start']]
    dens_end = max(k['end'] for k in dens) if dens else fork
    gam_end = max(k['end'] for k in gam) if gam else fork
    out = {'pre_fork_us': fork - t0, 'density_us': dens_end - fork, 'gametes_us': gam_end - fork,
           'exposed_us': (dens_end - fork) - (gam_end - fork), 'death_us': death['end'] - death['start'],
           'join_to_death_us': death['start'] - max(dens_end, gam_end),
           'density_kernels': [k['name'] for k in sorted(dens, key=lambda k: k['start'])],
           'gamete_kernels': [k['name'] for k in sorted(gam, key=lambda k: k['start'])]}
    if next_start is not None:
        out['step_us'] = next_start - t0
    return out


def power_limit_w():
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(0)
        return pynvml.nvmlDeviceGetEnforcedPowerLimit(h) / 1000.0
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--workload', default='c2')
    ap.add_argument('--presteps', type=int, default=600)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--out', required=True)
    args = ap.parse_args()

    import torch
    from torch.profiler import profile, ProfilerActivity
    import bench
    from geonomics_b200 import workloads, _lib

    cfg = dict(workloads.CONFIGS[args.workload])
    dev, w, _ = bench.make_species(cfg, 0)
    done = 0
    while done < args.presteps:
        c = min(64, args.presteps - done)
        dev.step(c)
        done += c
    dev.step(4)                                   # the captured graph is warm
    dev.sync()
    dev.step_records()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        dev.step(args.steps + 1)                  # + 1: the last step's length is the next step's start
        dev.sync()
        torch.cuda.synchronize()
    counters = dev.counters()
    recs = dev.step_records()
    dev.close()

    trace = os.path.join(tempfile.mkdtemp(prefix='gnx_timeline_'), 'trace.json')
    prof.export_chrome_trace(trace)
    with open(trace) as f:
        events = json.load(f)['traceEvents']
    acts = sorted(({'name': short_name(e['name']), 'kind': e['cat'],
                    'stream': e.get('args', {}).get('stream', e.get('tid')),
                    'start': float(e['ts']), 'end': float(e['ts']) + float(e['dur'])}
                   for e in events if e.get('cat') in ('kernel', 'gpu_memset', 'gpu_memcpy')), key=lambda k: k['start'])
    kernels = [a for a in acts if a['kind'] == 'kernel']
    steps = split_steps(kernels)
    rows = []
    gap_us = {}
    for s, ks in enumerate(steps):
        nxt = steps[s + 1][0]['start'] if s + 1 < len(steps) else None
        r = step_summary(ks, nxt)
        if r is not None and nxt is not None:
            others = [a for a in acts if a['kind'] != 'kernel' and ks[0]['start'] <= a['start'] < nxt]
            r['gaps'] = step_gaps(ks, others)
            for g in r['gaps']:
                gap_us.setdefault(g['after'] + ' -> ' + g['before'], []).append(g['us'])
            r['kernels'] = [{'name': k['name'], 'stream': k['stream'], 'start_us': k['start'] - ks[0]['start'],
                             'end_us': k['end'] - ks[0]['start']} for k in ks]
            r['non_kernel'] = [{'name': o['name'], 'kind': o['kind'], 'stream': o['stream'],
                                'start_us': o['start'] - ks[0]['start'], 'end_us': o['end'] - ks[0]['start']}
                               for o in others]
            rows.append(r)
    cells = w['land_dim'][0] * w['land_dim'][1]
    durs = {}
    for ks in steps:
        for k in ks:
            durs.setdefault(k['name'], []).append(k['end'] - k['start'])
    raster = {n: {'us_per_launch': float(np.median(durs[n])), 'bytes_per_launch': b * cells,
                  'GBs': b * cells / (np.median(durs[n]) * 1e-6) / 1e9}
              for n, b in RASTER_BYTES_PER_CELL.items() if n in durs}
    keys = ('pre_fork_us', 'density_us', 'gametes_us', 'exposed_us', 'death_us', 'join_to_death_us', 'step_us')
    out = {'workload': args.workload + ': ' + bench.workload_desc(cfg),
           'library': os.path.relpath(_lib.LIB_PATH, os.path.dirname(HERE)),
           'presteps': args.presteps, 'steps_traced': len(rows),
           'gpu': torch.cuda.get_device_name(0),
           'power_limit_w': power_limit_w(),
           'kernels_listed': len(kernels) > 0,
           'median': {k: float(np.median([r[k] for r in rows])) for k in keys} if rows else None,
           'min': {k: float(np.min([r[k] for r in rows])) for k in keys} if rows else None,
           'max': {k: float(np.max([r[k] for r in rows])) for k in keys} if rows else None,
           'kernel_median_us': {n: float(np.median(v)) for n, v in sorted(durs.items())},
           'gap_median_us': {n: float(np.median(v)) for n, v in sorted(gap_us.items())},
           'raster_bytes': raster,
           # (fix list, deferred list); libraries without k_raster_Nd keep no such lengths
           'density_lists_last_step': counters.get('density_lists') if 'k_raster_Nd' in durs else None,
           'population_last_step': int(recs[-1]['Nt']) if recs else None,
           'steps': rows}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ('workload', 'library', 'gpu', 'power_limit_w', 'steps_traced', 'median',
                                          'gap_median_us', 'density_lists_last_step')}))


if __name__ == '__main__':
    main()
